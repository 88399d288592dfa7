"""CPU: the recognizer's whole HOST flow (rows R4, R5, R10, R11 + orientation fallback + source_downscale) of the
product against the REFERENCE's own `TextRecognizer.__call__`.

The reference class is executed from the reference tree (oracle/refcheck.py: build_reference_recognizer_shell; its
uninstallable imports are stubs, ParseqDataset / data functions / tokenizer are the real files) with a stand-in PARSeq
whose output is a function of (crop pixels, padded width, mini-batch length); the product runs the same stand-in behind
its two device entry points (tests/flow_standins.py).  Equal contents / scores / directions / points therefore mean:
same crops, same bucketing order, same mini-batches and padding, same result pairing and order restoration, same
fallback decisions.  tests/golden/flow_ref.npz and tests/golden/live_ref.npz store the reference's outputs, so the
tests need no reference tree."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import flow_standins as FS  # noqa: E402
from oracle import build_crop_host  # noqa: E402


@pytest.fixture()
def device_crops_on_host(monkeypatch):
    """The device-crop path with its three device calls served by the product's crop arithmetic compiled for the host."""
    from yomitoku_b200 import models as M
    from yomitoku_b200.data import layout_crop_buffers
    host = ctypes.CDLL(build_crop_host.build())
    vp = ctypes.c_void_p

    class Buf:
        def __init__(self, arr):
            self.arr = arr

        def data_ptr(self):
            return self.arr.ctypes.data

    def extract(pages_dev, geoms, stream=None):
        sb, cb = layout_crop_buffers(geoms)
        scratch, canv = np.zeros(max(sb, 1), np.uint8), np.full(max(cb, 1), 99, np.uint8)
        pg = np.ascontiguousarray(pages_dev.numpy())
        host.crop_host_extract(pg.ctypes.data_as(vp), pg.shape[1], pg.shape[2], geoms.ctypes.data_as(vp), len(geoms),
                               scratch.ctypes.data_as(vp), canv.ctypes.data_as(vp))
        return Buf(canv), cb

    def halve(pages_dev, stream=None):
        src = np.ascontiguousarray(pages_dev.numpy())
        n, H, W, _ = src.shape
        dH, dW = int(np.rint(H * 0.5)), int(np.rint(W * 0.5))
        dst = np.zeros((n, dH, dW, 3), np.uint8)
        for i in range(n):
            host.crop_host_halve(src[i].ctypes.data_as(vp), W, H, dW, dH, dst[i].ctypes.data_as(vp))
        return torch.from_numpy(dst)

    monkeypatch.setattr(M, "extract_crops_device", extract)
    monkeypatch.setattr(M, "halve_pages_device", halve)
    monkeypatch.setattr(M, "concat_device_buffers", lambda parts, stream=None: parts[0][0] if len(parts) == 1 else
                        Buf(np.concatenate([t.arr[:n] for t, n in parts])))

    def enable(rec):
        rec.device_crops = True
        rec._upload_page = lambda img: torch.from_numpy(np.ascontiguousarray(img))[None]
        return rec
    return enable


def _same(res, contents, scores, directions):
    assert list(res.contents) == list(contents)
    assert list(res.directions) == list(directions)
    assert np.allclose(res.scores, scores, rtol=1e-6, atol=0)


@pytest.mark.parametrize("name", sorted(FS.CASES))
def test_product_flow_matches_reference_fixture(name, device_crops_on_host):
    z = np.load(os.path.join(HERE, "golden", "flow_ref.npz"), allow_pickle=True)
    contents, scores, directions = z[name + "_contents"].tolist(), z[name + "_scores"], z[name + "_directions"].tolist()
    assert len(contents) >= 1
    rec, page, quads = FS.product_recognizer(name)
    host_res, _ = rec(page, quads)                      # crops cut by OpenCV on the host
    _same(host_res, contents, scores, directions)
    dev_res, _ = device_crops_on_host(rec)(page, quads)     # crops cut by the device arithmetic
    _same(dev_res, contents, scores, directions)
    assert host_res.points == dev_res.points


@pytest.mark.parametrize("name", ["dynw_bucketing", "dropped_quad", "fallback_and_downscale"])
def test_product_flow_matches_reference_live(name):
    """The product's host-crop path against the reference's contents / scores / directions AND points (stored by
    tests/golden/make_golden_live.py)."""
    z = np.load(os.path.join(HERE, "golden", "live_ref.npz"))
    rec, page, quads = FS.product_recognizer(name)
    p, _ = rec(page, quads)
    _same(p, z["flow_%s_contents" % name].tolist(), z["flow_%s_scores" % name],
          z["flow_%s_directions" % name].tolist())
    assert p.points == z["flow_%s_points" % name].tolist()


def test_detector_flow_matches_reference_fixture():
    """Rows R1 (host pre-processing: flip, float32 INTER_AREA / linear resize to the floor-32 size, standardisation) and R3
    through `TextDetector.__call__`: quads and scores the reference's own TextDetector produced with the stand-in model."""
    z = np.load(os.path.join(HERE, "golden", "detflow_ref.npz"))
    det = FS.product_detector()
    for i, page in enumerate(FS.detector_pages()):
        res, vis = det(page)
        assert vis is None and len(res.points) > 50
        assert res.points == z["points%d" % i].tolist()
        assert res.scores == z["scores%d" % i].tolist()


def test_detector_flow_matches_reference_live():
    """TextDetector.preprocess (shape, sums, a seeded sample of the tensor: bit-equal) and __call__ against the
    reference's own TextDetector with the stand-in model (stored by tests/golden/make_golden_live.py)."""
    sys.path.insert(0, os.path.join(HERE, "golden"))
    from make_golden_live import PRE_SAMPLE, sample_index
    z = np.load(os.path.join(HERE, "golden", "live_ref.npz"))
    det = FS.product_detector()
    for i, page in enumerate(FS.detector_pages()):
        x = det.preprocess(page)
        assert tuple(x.shape) == tuple(z["detflow%d_pre_shape" % i])
        got = x.reshape(-1)[torch.from_numpy(sample_index(x.numel(), PRE_SAMPLE, 200 + i))].numpy()
        assert np.array_equal(got, z["detflow%d_pre_sample" % i])
        assert np.allclose([float(x.double().sum()), float((x.double() ** 2).sum())], z["detflow%d_pre_sum" % i],
                           rtol=1e-10, atol=0)
        p, _ = det(page)
        assert p.points == z["detflow%d_points" % i].tolist() and p.scores == z["detflow%d_scores" % i].tolist()
