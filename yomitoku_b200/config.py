"""Model configs for the hot path: the reference's dataclass defaults restated as plain nested dicts with attribute
access, plus YAML override merge.

Mirrors reference src/yomitoku/base.py:15-33 (load_yaml_config / load_config; OmegaConf there, absent in this image)
and the values of src/yomitoku/configs/cfg_text_detector_dbnet{,_v2,_v2_1}.py and
cfg_text_recognizer_parseq{,_v2,_small,_tiny,_large_v4_1,_tiny_dynw_v4}.py.  Only what the path reads is kept.
"""
import copy
import os
from pathlib import Path

import yaml

PKG_DIR = os.path.dirname(os.path.abspath(__file__))


class Config(dict):
    """dict with attribute access (cfg.data.batch_size) and getattr-with-default semantics like OmegaConf nodes."""

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError:
            raise AttributeError(key)

    def __setattr__(self, key, value):
        self[key] = value

    def __deepcopy__(self, memo):
        return Config({k: copy.deepcopy(v, memo) for k, v in self.items()})


def to_config(obj):
    if isinstance(obj, dict):
        return Config({k: to_config(v) for k, v in obj.items()})
    if isinstance(obj, (list, tuple)):
        return [to_config(v) for v in obj]
    return obj


def merge(base, override):
    """Deep merge `override` into a copy of `base` (OmegaConf.merge semantics for dict nodes; lists replace)."""
    out = copy.deepcopy(base)
    for k, v in (override or {}).items():
        if isinstance(v, dict) and isinstance(out.get(k), dict):
            out[k] = merge(out[k], v)
        else:
            out[k] = to_config(v)
    return out


def load_yaml_config(path_config):
    path_config = Path(path_config)
    if not path_config.exists():
        raise FileNotFoundError(f"Config file not found: {path_config}")
    with open(path_config, "r", encoding="utf-8") as f:
        return yaml.safe_load(f) or {}


def load_config(default_config, path_config=None):
    cfg = to_config(default_config() if callable(default_config) else default_config)
    if path_config is not None:
        cfg = merge(cfg, load_yaml_config(path_config))
    return cfg


# ------------------------------------------------------------------------------------------------ detector
def _dbnet(repo, thresh, box_thresh, unclip_ratio):
    return lambda: {
        "hf_hub_repo": repo,
        "backbone": {"name": "resnet50", "dilation": True},
        "decoder": {"in_channels": [256, 512, 1024, 2048], "hidden_dim": 256, "adaptive": True, "serial": True,
                    "smooth": False, "k": 50},
        "data": {"shortest_size": 1280, "limit_size": 1600},
        "post_process": {"min_size": 2, "thresh": thresh, "box_thresh": box_thresh, "max_candidates": 1500,
                         "unclip_ratio": unclip_ratio},
        "visualize": {"color": [0, 255, 0], "heatmap": False},
    }


TextDetectorDBNetConfig = _dbnet("KotaroKinoshita/yomitoku-text-detector-dbnet-open-beta", 0.15, 0.5, 7.0)
TextDetectorDBNetV2Config = _dbnet("KotaroKinoshita/yomitoku-text-detector-dbnet-v2", 0.2, 0.5, 5.0)
TextDetectorDBNetV2_1Config = _dbnet("KotaroKinoshita/yomitoku-text-detector-dbnet-v2_1", 0.3, 0.4, 3.5)


# ------------------------------------------------------------------------------------------------ recognizer
def _parseq(repo, charset, num_tokens, embed_dim, enc_heads, depth, patch, img_size=(32, 800), max_label_length=100,
            dec_heads=8, batch_size=128, font="MPLUS1p-Medium.ttf", extra_data=None):
    def make():
        data = {"num_workers": 4, "batch_size": batch_size, "img_size": list(img_size)}
        data.update(extra_data or {})
        return {
            "hf_hub_repo": repo,
            "charset": os.path.join(PKG_DIR, "resource", charset),
            "num_tokens": num_tokens,
            "max_label_length": max_label_length,
            "decode_ar": 1,
            "refine_iters": 1,
            "rec_orientation_fallback": False,
            "rec_orientation_fallback_thresh": 0.75,
            "data": data,
            "encoder": {"patch_size": list(patch), "num_heads": enc_heads, "embed_dim": embed_dim, "mlp_ratio": 4,
                        "depth": depth},
            "decoder": {"embed_dim": embed_dim, "num_heads": dec_heads, "mlp_ratio": 4, "depth": 1},
            "visualize": {"font": os.path.join(PKG_DIR, "resource", font), "color": [0, 0, 255], "font_size": 18},
        }
    return make


_R = "KotaroKinoshita/yomitoku-text-recognizer-"
TextRecognizerPARSeqConfig = _parseq(_R + "parseq-open-beta", "charset.txt", 7312, 512, 8, 12, (8, 8))
TextRecognizerPARSeqV2Config = _parseq(_R + "parseq-middle-v2", "charset.txt", 7312, 512, 8, 12, (8, 8))
TextRecognizerPARSeqSmallConfig = _parseq(_R + "parseq-small-open-beta", "charset.txt", 7312, 384, 8, 9, (16, 16))
TextRecognizerPARSeqTinyConfig = _parseq("KotaroKinoshita/yomitoku-text-recognizer-parseq-tiny", "charsetv2.txt", 7121,
                                         368, 8, 12, (8, 16), img_size=(32, 400), max_label_length=50,
                                         font="ShipporiMinchoB1-Bold.ttf")
TextRecognizerPARSeqLargeV41Config = _parseq(_R + "parseq-large-v4_1", "charsetv2.txt", 7121, 768, 8, 12, (8, 8),
                                             font="ShipporiMinchoB1-Bold.ttf")
TextRecognizerPARSeqTinyDynwV4Config = _parseq(_R + "parseq-tiny-dynw-v4", "charsetv2.txt", 7121, 192, 6, 12, (4, 8),
                                               dec_heads=6, batch_size=10, font="ShipporiMinchoB1-Bold.ttf",
                                               extra_data={"width_budget": 8000, "max_batch_size": 64})


# ------------------------------------------------------------------------------------------------ layout models
def _rtdetr(repo, num_classes, thresh_score, category, role=None, img=640, num_queries=300):
    """Values of reference configs/cfg_layout_parser_rtdtrv2{,_v2}.py, cfg_table_structure_recognizer_rtdtrv2.py and
    cfg_table_cell_parser_rtdtrv2.py."""
    def make():
        cfg = {
            "hf_hub_repo": repo,
            "thresh_score": thresh_score,
            "data": {"img_size": [img, img]},
            "PResNet": {"depth": 50, "variant": "d", "freeze_at": 0, "return_idx": [1, 2, 3], "num_stages": 4,
                        "freeze_norm": True},
            "HybridEncoder": {"in_channels": [512, 1024, 2048], "feat_strides": [8, 16, 32], "hidden_dim": 256,
                              "use_encoder_idx": [2], "num_encoder_layers": 1, "nhead": 8, "dim_feedforward": 1024,
                              "dropout": 0.0, "enc_act": "gelu", "expansion": 1.0, "depth_mult": 1, "act": "silu"},
            "RTDETRTransformerv2": {"num_classes": num_classes, "feat_channels": [256, 256, 256],
                                    "feat_strides": [8, 16, 32], "hidden_dim": 256, "num_levels": 3, "num_layers": 6,
                                    "num_queries": num_queries, "num_denoising": 100, "label_noise_ratio": 0.5,
                                    "box_noise_scale": 1.0, "eval_spatial_size": [img, img], "eval_idx": -1,
                                    "num_points": [4, 4, 4], "cross_attn_method": "default",
                                    "query_select_method": "default"},
            "category": list(category),
        }
        if role is not None:
            cfg["role"] = list(role)
        return cfg
    return make


_LAYOUT_CATEGORY = ["tables", "figures", "paragraphs", "section_headings", "page_header", "page_footer"]
_LAYOUT_ROLE = ["section_headings", "page_header", "page_footer"]
LayoutParserRTDETRv2Config = _rtdetr("KotaroKinoshita/yomitoku-layout-parser-rtdtrv2-open-beta", 6, 0.5,
                                     _LAYOUT_CATEGORY, _LAYOUT_ROLE)
LayoutParserRTDETRv2V2Config = _rtdetr("KotaroKinoshita/yomitoku-layout-parser-rtdtrv2-v2", 6, 0.5, _LAYOUT_CATEGORY,
                                       _LAYOUT_ROLE)
TableStructureRecognizerRTDETRv2Config = _rtdetr(
    "KotaroKinoshita/yomitoku-table-structure-recognizer-rtdtrv2-open-beta", 3, 0.4, ["row", "col", "span"])
# the cell detector was trained with 900 queries; it runs 1500 at inference (the weights do not depend on the count) so
# that dense tables of up to ~1000 cells stay below the detection limit
TableCellParserRTDETRv2Config = _rtdetr("KotaroKinoshita/yomitoku-cell-detector-rtdtrv2-v1", 6, 0.5,
                                        ["table", "cell", "header", "empty", "kv_item", "grid"], img=960,
                                        num_queries=1500)
