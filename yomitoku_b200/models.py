"""Device-backed DBNet and PARSeq model objects: the `self.model` of TextDetector / TextRecognizer.

They keep the surface the reference's modules touch from outside (SURVEY.md section 8b "model-level seam"):
`model(tensor)`, `.eval()`, `.to(device)`, `.state_dict()/.load_state_dict()` (reference key set, Appendix C),
`.from_pretrained(repo, cfg=cfg)`, `PARSeq.tokenizer`, `PARSeq.refine_iters`, `PARSeq.export_onnx` - but the forward
pass is the hand-written sm_100a engine behind the C ABI (include/yomitoku_b200.h).  There is no CPU fallback: a
forward without the CUDA library and a GPU raises.

Reference: src/yomitoku/models/dbnet_plus.py:233-246, src/yomitoku/models/parseq.py:49-311.
"""
import ctypes
import math
import threading
from collections import OrderedDict

import numpy as np
import torch

from . import _lib


def _stream_ptr(stream):
    """torch.cuda.Stream (or None = default stream) -> cudaStream_t for the C ABI."""
    return None if stream is None else ctypes.c_void_p(stream.cuda_stream)


def _he_conv(g, cout, cin, kh, kw, gain=1.0):
    return torch.randn(cout, cin, kh, kw, generator=g) * (gain * math.sqrt(2.0 / (cin * kh * kw)))


class _DeviceModel:
    """Minimal nn.Module-like shell around a C handle."""

    def __init__(self):
        self._sd = None
        self._handle = None
        self._device = torch.device("cpu")
        self.training = False

    def eval(self):
        self.training = False
        return self

    def to(self, device):
        """Like nn.Module.to(device): the C handle is created on (and bound to) this device.  Moving an already
        materialised model drops the handle; the next forward re-creates it on the new device."""
        new = torch.device(device) if not isinstance(device, torch.device) else device
        if new != self._device:
            self._release()
        self._device = new
        return self

    def cuda_device(self):
        """torch.device the device calls run on: the one given to `.to()`, or the thread's current CUDA device when the
        model was never moved (`cuda` without an index means the current device, as in torch)."""
        if self._device.type == "cuda" and self._device.index is not None:
            return self._device
        return torch.device("cuda", torch.cuda.current_device())

    def state_dict(self):
        return OrderedDict(self._sd)

    def load_state_dict(self, sd, strict=True):
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        if strict and (missing or unexpected):
            raise RuntimeError("Error(s) in loading state_dict: missing %s unexpected %s" % (missing[:5], unexpected[:5]))
        for k in self._sd:
            if k in sd:
                if tuple(sd[k].shape) != tuple(self._sd[k].shape):
                    raise RuntimeError("size mismatch for %s" % k)
                self._sd[k] = sd[k].detach().clone()
        self._release()
        return self

    def parameters(self):
        return (v for v in self._sd.values() if torch.is_floating_point(v))

    def _release(self):
        raise NotImplementedError

    def _require_cuda(self):
        if not torch.cuda.is_available():
            raise _lib.YtkError(
                "%s runs only on a CUDA device (sm_100a): no GPU is visible and there is no CPU fallback on the "
                "hot path" % type(self).__name__)

    @classmethod
    def from_pretrained(cls, repo, cfg=None, **kw):
        """Loads the reference's HF `model.safetensors` (strict state_dict keys).  Offline (no hub cache) this raises
        like huggingface_hub does."""
        from huggingface_hub import hf_hub_download
        from safetensors.torch import load_file
        path = hf_hub_download(repo, "model.safetensors")
        m = cls(cfg=cfg)
        m.load_state_dict(load_file(path), strict=True)
        return m


def extract_crops_device(pages_dev, geoms, stream=None):
    """Device-side crop extraction (C ABI ytk_extract_crops_u8, csrc/crop_ops.cu).

    pages_dev: (n, H0, W0, 3) uint8 BGR cuda tensor; geoms: CROP_GEOM_DTYPE records (data.crop_geometry) - their
    roi_off / pix_off are (re)assigned here, crops packed back to back in record order.  Returns (canvases, total
    bytes): a flat uint8 cuda tensor holding every crop's (canvas_h, canvas_w, 3) RGB canvas at geoms["pix_off"], ready
    for PARSeq.run_packed_ptr(..., on_device=1).  Asynchronous on `stream` (default: the current stream)."""
    from .data import CROP_GEOM_DTYPE, layout_crop_buffers
    if not (isinstance(pages_dev, torch.Tensor) and pages_dev.is_cuda and pages_dev.dtype == torch.uint8
            and pages_dev.dim() == 4 and pages_dev.shape[3] == 3 and pages_dev.is_contiguous()):
        raise ValueError("extract_crops_device: pages_dev must be a contiguous (n, H, W, 3) uint8 cuda tensor")
    if not (isinstance(geoms, np.ndarray) and geoms.dtype == CROP_GEOM_DTYPE and geoms.flags.c_contiguous):
        raise ValueError("extract_crops_device: geoms must be a contiguous CROP_GEOM_DTYPE array")
    scratch_bytes, total = layout_crop_buffers(geoms)      # writes roi_off / pix_off into the caller's records
    ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.device(pages_dev.device)
    # scratch = ROIs + (16-byte aligned) the device copy of the records (include/yomitoku_b200.h)
    scratch_bytes = (scratch_bytes + 15) // 16 * 16 + geoms.nbytes
    with ctx:
        scratch = torch.empty(max(scratch_bytes, 1), dtype=torch.uint8, device=pages_dev.device)
        canv = torch.empty(max(total, 1), dtype=torch.uint8, device=pages_dev.device)
    n, H0, W0, _ = pages_dev.shape
    _lib.check(_lib.lib().ytk_extract_crops_u8(pages_dev.data_ptr(), n, H0, W0, geoms.ctypes.data, len(geoms),
                                               scratch.data_ptr(), scratch_bytes, canv.data_ptr(), total,
                                               _stream_ptr(stream)))
    if stream is not None:
        # the scratch buffer is only read by the canvas kernel queued on `stream`: hand it back to the allocator in
        # stream order
        scratch.record_stream(stream)
    return canv, total


DB_RUN_DTYPE = np.dtype([("root", "<i4"), ("y", "<i4"), ("x0", "<i4"), ("x1", "<i4"), ("sum", "<f8")])   # = ytk_db_run


_POST_BUFS = {}                      # (device, n, H, W, max_runs) -> device scratch + page-locked staging, reused
_POST_LOCK = threading.Lock()


def dbnet_post_front(prob_dev, thresh, stream=None, max_runs=32768):
    """Device-side front half of the DBNet post-processing (C ABI ytk_dbnet_post_front, csrc/dbpost_ops.cu):
    prob_dev (n, H, W) fp32 cuda -> per page either a DB_RUN_DTYPE array (the row runs of the 8-connected components of
    prob > thresh, input of DBnetPostProcessor.boxes_from_runs) or None when the page has to take the host path
    (a component with a hole, which OpenCV reports as an extra contour, or more than `max_runs` runs).  Only the runs
    (24 bytes each; a 200-line page has ~4 k) cross PCIe instead of the 7.6 MB map.  Synchronises `stream`.
    Returns (runs per page, meta (n, 4) int32 = {runs, components, 4 x Euler number, overflow})."""
    if not (isinstance(prob_dev, torch.Tensor) and prob_dev.is_cuda and prob_dev.dtype == torch.float32
            and prob_dev.dim() == 3 and prob_dev.is_contiguous()):
        raise ValueError("dbnet_post_front: prob_dev must be a contiguous (n, H, W) float32 cuda tensor")
    n, H, W = prob_dev.shape
    dev = prob_dev.device
    rec = DB_RUN_DTYPE.itemsize
    with _POST_LOCK, (torch.cuda.stream(stream) if stream is not None else torch.cuda.device(dev)):
        key = (dev.index, n, H, W, max_runs)
        bufs = _POST_BUFS.get(key)
        if bufs is None:
            # scratch of the kernels + page-locked landing zone of the results: allocated once per batch shape (a
            # cudaHostAlloc per call would serialise against the other streams of the pipeline)
            bufs = (torch.empty((n, H, W), dtype=torch.int32, device=dev),
                    torch.empty((n, max_runs, rec), dtype=torch.uint8, device=dev),
                    torch.empty((n, 4), dtype=torch.int32, device=dev),
                    torch.empty((n, max_runs, rec), dtype=torch.uint8, pin_memory=True),
                    torch.empty((n, 4), dtype=torch.int32, pin_memory=True))
            if len(_POST_BUFS) >= 4:
                _POST_BUFS.pop(next(iter(_POST_BUFS)))
            _POST_BUFS[key] = bufs
        labels, runs, meta, runs_h, meta_h = bufs
        cur = torch.cuda.current_stream(dev)
        _lib.check(_lib.lib().ytk_dbnet_post_front(prob_dev.data_ptr(), n, H, W, float(thresh), labels.data_ptr(),
                                                   labels.numel() * 4, runs.data_ptr(), max_runs, meta.data_ptr(),
                                                   ctypes.c_void_p(cur.cuda_stream)))
        meta_h.copy_(meta, non_blocking=True)
        cur.synchronize()
        m = meta_h.numpy().copy()
        ok = [not (int(m[i, 3]) or int(m[i, 0]) > max_runs or int(m[i, 1]) * 4 != int(m[i, 2])) for i in range(n)]
        for i in range(n):
            if ok[i] and m[i, 0]:
                runs_h[i, :int(m[i, 0])].copy_(runs[i, :int(m[i, 0])], non_blocking=True)
        cur.synchronize()
        out = [runs_h[i, :int(m[i, 0])].numpy().reshape(-1).view(DB_RUN_DTYPE).copy() if ok[i] else None
               for i in range(n)]
    return out, m


def halve_pages_device(pages_dev, stream=None):
    """One level of the source_downscale pyramid on the GPU (C ABI ytk_halve_pages_u8): (n, H, W, 3) uint8 cuda tensor ->
    (n, cvRound(H / 2), cvRound(W / 2), 3), equal to cv2.resize(page, None, fx=0.5, fy=0.5, INTER_AREA) per page."""
    n, H, W, _ = pages_dev.shape
    dH, dW = int(np.rint(H * 0.5)), int(np.rint(W * 0.5))      # round half to even, like cvRound
    if dH < 1 or dW < 1:
        raise ValueError("halve_pages_device: a %dx%d page cannot be halved" % (H, W))
    ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.device(pages_dev.device)
    with ctx:
        out = torch.empty((n, dH, dW, 3), dtype=torch.uint8, device=pages_dev.device)
    _lib.check(_lib.lib().ytk_halve_pages_u8(pages_dev.data_ptr(), n, H, W, out.data_ptr(), dH, dW, _stream_ptr(stream)))
    return out


def extract_crops_pyramid(pages, geoms, levels, stream=None):
    """`extract_crops_device` for records that live on different pyramid levels (source_downscale).  pages: dict
    level -> (n, H_k, W_k, 3) cuda tensor; missing levels are built on demand by halving the level below (the dict is
    filled in place).  geoms / levels: records in packing order and their levels.  Returns (canvases, total bytes,
    pix_off): one flat buffer, and every record's canvas offset in it (one extraction per level, back to back)."""
    levels = np.asarray(levels, np.int64)
    n = len(geoms)
    pix_off = np.zeros(n, np.int64)
    parts, base = [], 0
    for k in sorted(set(levels.tolist())):
        for j in range(1, k + 1):
            if j not in pages:
                pages[j] = halve_pages_device(pages[j - 1], stream)
        idx = np.nonzero(levels == k)[0]
        sub = np.ascontiguousarray(geoms[idx])
        canv, total = extract_crops_device(pages[k], sub, stream)
        pix_off[idx] = base + sub["pix_off"]
        parts.append((canv, total))
        base += total
    if not parts:
        raise ValueError("extract_crops_pyramid: no records")
    return concat_device_buffers(parts, stream), base, pix_off


def plan_crop_offsets(geoms, levels):
    """Host-only twin of `extract_crops_pyramid`'s packing: (total bytes, pix_off per record) of the buffer it will
    produce for these records (one block per pyramid level in ascending order, canvases back to back inside a block)."""
    levels = np.asarray(levels, np.int64)
    pix_off = np.zeros(len(geoms), np.int64)
    base = 0
    for k in sorted(set(levels.tolist())):
        idx = np.nonzero(levels == k)[0]
        size = geoms["canvas_w"][idx].astype(np.int64) * geoms["canvas_h"][idx] * 3
        pix_off[idx] = base + np.cumsum(size) - size
        base += int(size.sum())
    return base, pix_off


def concat_device_buffers(parts, stream=None):
    """parts: list of (flat uint8 cuda tensor, used bytes) -> one flat uint8 tensor holding them back to back (the
    copy is queued on `stream`, like the kernels that filled the parts)."""
    if len(parts) == 1:
        return parts[0][0]
    if stream is not None:
        with torch.cuda.stream(stream):
            return torch.cat([t[:n] for t, n in parts])
    return torch.cat([t[:n] for t, n in parts])


# ======================================================================================================== DBNet
def _dbnet_random_state_dict(seed=0):
    """Random init with the reference's key set (DBNet(cfg) with from_pretrained=False, base.py:84-86)."""
    g = torch.Generator().manual_seed(seed)
    sd = OrderedDict()

    def bn(p, c):
        sd[p + ".weight"] = torch.ones(c)
        sd[p + ".bias"] = torch.full((c,), 1e-4)
        sd[p + ".running_mean"] = torch.zeros(c)
        sd[p + ".running_var"] = torch.ones(c)
        sd[p + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)

    b = "backbone.body."
    sd[b + "conv1.weight"] = _he_conv(g, 64, 3, 7, 7)
    bn(b + "bn1", 64)
    inpl = 64
    for li, (pl, nb) in enumerate(((64, 3), (128, 4), (256, 6), (512, 3)), start=1):
        for i in range(nb):
            q = "%slayer%d.%d." % (b, li, i)
            sd[q + "conv1.weight"] = _he_conv(g, pl, inpl, 1, 1)
            bn(q + "bn1", pl)
            sd[q + "conv2.weight"] = _he_conv(g, pl, pl, 3, 3)
            bn(q + "bn2", pl)
            sd[q + "conv3.weight"] = _he_conv(g, pl * 4, pl, 1, 1, 0.5)
            bn(q + "bn3", pl * 4)
            if i == 0:
                sd[q + "downsample.0.weight"] = _he_conv(g, pl * 4, inpl, 1, 1, 0.7)
                bn(q + "downsample.1", pl * 4)
            inpl = pl * 4
    d = "decoder."
    for i, c in enumerate((256, 512, 1024, 2048), start=1):
        sd["%sinput_proj.layer%d.weight" % (d, i)] = _he_conv(g, 256, c, 1, 1, 0.7)
    sd[d + "out_proj.layer1.weight"] = _he_conv(g, 64, 256, 3, 3)
    for i in (2, 3, 4):
        sd["%sout_proj.layer%d.0.weight" % (d, i)] = _he_conv(g, 64, 256, 3, 3)
    for name, cin in (("binarize", 256), ("thresh", 257)):
        q = d + name + "."
        sd[q + "0.weight"] = _he_conv(g, 64, cin, 3, 3)
        bn(q + "1", 64)
        sd[q + "3.weight"] = torch.randn(64, 64, 2, 2, generator=g) * math.sqrt(2.0 / 64)
        sd[q + "3.bias"] = torch.zeros(64)
        bn(q + "4", 64)
        sd[q + "6.weight"] = torch.randn(64, 1, 2, 2, generator=g) * math.sqrt(2.0 / 64)
        sd[q + "6.bias"] = torch.zeros(1)
    a = d + "concat_attention."
    sd[a + "conv.weight"] = _he_conv(g, 64, 256, 3, 3)
    sd[a + "conv.bias"] = torch.zeros(64)
    e = a + "enhanced_attention."
    sd[e + "channel_wise.1.weight"] = _he_conv(g, 16, 64, 1, 1)
    sd[e + "channel_wise.3.weight"] = _he_conv(g, 64, 16, 1, 1)
    sd[e + "spatial_wise.0.weight"] = torch.randn(1, 1, 3, 3, generator=g) * 0.5
    sd[e + "spatial_wise.2.weight"] = torch.randn(1, 1, 1, 1, generator=g)
    sd[e + "attention_wise.0.weight"] = _he_conv(g, 4, 64, 1, 1)
    return sd


class DBNet(_DeviceModel):
    """reference models/dbnet_plus.py:233-246.  `model(tensor)` takes the normalised (1,3,H,W) fp32 tensor of
    TextDetector.preprocess and returns OrderedDict(binary=(1,1,H,W) fp32 probabilities)."""

    def __init__(self, cfg=None, seed=0):
        super().__init__()
        self.cfg = cfg
        self._sd = _dbnet_random_state_dict(seed)
        self._shortest = int(cfg.data.shortest_size) if cfg is not None else 1280
        self._limit = int(cfg.data.limit_size) if cfg is not None else 1600

    # -- handle management
    def _ensure(self):
        self._require_cuda()
        if self._handle is None:
            L = _lib.lib()
            tab, keep = _lib.tensor_table(self._sd)
            h = ctypes.c_void_p()
            with torch.cuda.device(self.cuda_device()):     # the handle binds to the device current at create()
                _lib.check(L.ytk_dbnet_create(tab, len(tab), self._shortest, self._limit, ctypes.byref(h)))
            self._handle = h
        return self._handle

    def _release(self):
        if self._handle is not None:
            _lib.lib().ytk_dbnet_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def input_size(self, h, w):
        """(Hn, Wn) the network sees for an h x w page = reference resize_shortest_edge (functions.py:212-224)."""
        from .data import shortest_edge_size
        return shortest_edge_size(h, w, self._shortest, self._limit)

    def __call__(self, tensor):
        return self.forward(tensor)

    def forward(self, tensor):
        """Model-level seam: (N,3,H,W) fp32 (host or cuda) -> {"binary": (N,1,H,W) fp32 on the same device}."""
        h = self._ensure()
        if tensor.dim() != 4 or tensor.shape[1] != 3:
            raise ValueError("DBNet expects (N,3,H,W), got %s" % (tuple(tensor.shape),))
        n, _, H, W = tensor.shape
        x = tensor.detach().to(torch.float32).contiguous()
        on_dev = x.is_cuda
        out = torch.empty((n, 1, H, W), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().ytk_dbnet_forward_f32(h, x.data_ptr(), 1 if on_dev else 0, n, H, W, out.data_ptr(),
                                                    1 if on_dev else 0, None))
        return OrderedDict(binary=out)

    def detect_pages_u8(self, pages, out=None, stream=None):
        """Fused fast path: pages (n,H0,W0,3) uint8 BGR (numpy / torch, host or cuda) -> (n,Hn,Wn) fp32 probability
        maps (pre-processing runs on the GPU).  Pages that would be up-scaled need the model-level seam."""
        h = self._ensure()
        t = pages if isinstance(pages, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(pages))
        if t.dim() == 3:
            t = t[None]
        t = t.contiguous()
        n, H0, W0, _ = t.shape
        Hn, Wn = self.input_size(H0, W0)
        if out is None:
            out = torch.empty((n, Hn, Wn), dtype=torch.float32, device=t.device,
                              pin_memory=(not t.is_cuda) and torch.cuda.is_available())
        _lib.check(_lib.lib().ytk_dbnet_forward_u8(h, t.data_ptr(), 1 if t.is_cuda else 0, n, H0, W0, out.data_ptr(),
                                                   1 if out.is_cuda else 0, _stream_ptr(stream)))
        return out

    def flops(self, n, Hn, Wn):
        return _lib.lib().ytk_dbnet_flops(self._ensure(), n, Hn, Wn)


# ======================================================================================================== PARSeq
def _parseq_random_state_dict(cfg, seed=0):
    """Random init with the reference's key set and init scheme (parseq.py:28-46,81-82: trunc-normal(0.02) linears /
    embeddings, ones/zeros norms; encoder = timm ViT defaults)."""
    g = torch.Generator().manual_seed(seed)
    D = cfg.encoder.embed_dim
    ph, pw = cfg.encoder.patch_size
    gh, gw = cfg.data.img_size[0] // ph, cfg.data.img_size[1] // pw
    depth, r = cfg.encoder.depth, cfg.encoder.mlp_ratio
    S = cfg.max_label_length + 1

    def tn(*shape):
        return torch.randn(*shape, generator=g).clamp_(-2, 2) * 0.02

    sd = OrderedDict()
    e = "encoder."
    sd[e + "pos_embed"] = tn(1, gh * gw, D)
    sd[e + "patch_embed.proj.weight"] = torch.randn(D, 3, ph, pw, generator=g) * math.sqrt(1.0 / (3 * ph * pw))
    sd[e + "patch_embed.proj.bias"] = torch.zeros(D)
    for i in range(depth):
        p = "%sblocks.%d." % (e, i)
        sd[p + "norm1.weight"], sd[p + "norm1.bias"] = torch.ones(D), torch.zeros(D)
        sd[p + "attn.qkv.weight"], sd[p + "attn.qkv.bias"] = tn(3 * D, D), torch.zeros(3 * D)
        sd[p + "attn.proj.weight"], sd[p + "attn.proj.bias"] = tn(D, D), torch.zeros(D)
        sd[p + "norm2.weight"], sd[p + "norm2.bias"] = torch.ones(D), torch.zeros(D)
        sd[p + "mlp.fc1.weight"], sd[p + "mlp.fc1.bias"] = tn(r * D, D), torch.zeros(r * D)
        sd[p + "mlp.fc2.weight"], sd[p + "mlp.fc2.bias"] = tn(D, r * D), torch.zeros(D)
    sd[e + "norm.weight"], sd[e + "norm.bias"] = torch.ones(D), torch.zeros(D)
    p = "decoder.layers.0."
    for att in ("self_attn", "cross_attn"):
        sd[p + att + ".in_proj_weight"] = torch.randn(3 * D, D, generator=g) * math.sqrt(2.0 / (4 * D))
        sd[p + att + ".in_proj_bias"] = torch.zeros(3 * D)
        sd[p + att + ".out_proj.weight"], sd[p + att + ".out_proj.bias"] = tn(D, D), torch.zeros(D)
    H = cfg.decoder.mlp_ratio * D
    sd[p + "linear1.weight"], sd[p + "linear1.bias"] = tn(H, D), torch.zeros(H)
    sd[p + "linear2.weight"], sd[p + "linear2.bias"] = tn(D, H), torch.zeros(D)
    for n in ("norm1", "norm2", "norm_q", "norm_c"):
        sd[p + n + ".weight"], sd[p + n + ".bias"] = torch.ones(D), torch.zeros(D)
    sd["decoder.norm.weight"], sd["decoder.norm.bias"] = torch.ones(D), torch.zeros(D)
    sd["head.weight"], sd["head.bias"] = tn(cfg.num_tokens - 2, D), torch.zeros(cfg.num_tokens - 2)
    sd["text_embed.embedding.weight"] = tn(cfg.num_tokens, D)
    sd["pos_queries"] = tn(1, S, D)
    return sd


class PARSeq(_DeviceModel):
    """reference models/parseq.py:49-311.  `model(images)` takes (B,3,32,W) fp32 in [-1,1] and returns logits
    (B, S, C); `recognize_crops` is the fused ragged path that returns only (ids, probs)."""

    def __init__(self, cfg=None, seed=0):
        super().__init__()
        self.cfg = cfg
        self.max_label_length = cfg.max_label_length
        self.decode_ar = cfg.decode_ar
        self._refine_iters = int(cfg.refine_iters)
        self.export_onnx = False
        self.tokenizer = None
        self.repetition_stop = bool(getattr(cfg, "repetition_stop", True))
        self.rep_period_max = int(getattr(cfg, "rep_period_max", 8))
        self.rep_min_run_p1 = int(getattr(cfg, "rep_min_run_p1", 8))
        self.rep_min_repeats = int(getattr(cfg, "rep_min_repeats", 3))
        self._sd = _parseq_random_state_dict(cfg, seed)

    def __setattr__(self, name, value):
        # the repetition-stop knobs and decode_ar are baked into the C handle at creation: changing one afterwards (the
        # reference reads them from the module at every forward, models/parseq.py:93-96,189) drops the handle so that
        # the next forward re-creates it with the new values instead of silently keeping the old ones
        if name in ("repetition_stop", "rep_period_max", "rep_min_run_p1", "rep_min_repeats", "decode_ar") and \
                getattr(self, "_handle", None) is not None and getattr(self, name, value) != value:
            self._release()
        object.__setattr__(self, name, value)

    @property
    def refine_iters(self):
        return self._refine_iters

    @refine_iters.setter
    def refine_iters(self, v):
        self._refine_iters = int(v)
        if self._handle is not None:
            _lib.lib().ytk_parseq_set_refine_iters(self._handle, self._refine_iters)

    @property
    def num_classes(self):
        return self.cfg.num_tokens - 2

    def _ensure(self):
        self._require_cuda()
        if self._handle is None:
            c = self.cfg
            L = _lib.lib()
            tab, keep = _lib.tensor_table(self._sd)
            cc = _lib.YtkParseqCfg(c.encoder.embed_dim, c.encoder.num_heads, c.encoder.depth, c.encoder.patch_size[0],
                                   c.encoder.patch_size[1], c.data.img_size[0], c.data.img_size[1], c.num_tokens,
                                   c.max_label_length, c.decoder.num_heads, c.encoder.mlp_ratio, c.decoder.mlp_ratio,
                                   self._refine_iters, 1 if self.repetition_stop else 0, self.rep_period_max,
                                   self.rep_min_run_p1, self.rep_min_repeats, 1 if self.decode_ar else 0)
            h = ctypes.c_void_p()
            with torch.cuda.device(self.cuda_device()):     # the handle binds to the device current at create()
                _lib.check(L.ytk_parseq_create(tab, len(tab), ctypes.byref(cc), ctypes.byref(h)))
            self._handle = h
        return self._handle

    def _release(self):
        if self._handle is not None:
            _lib.lib().ytk_parseq_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def __call__(self, images, max_length=None):
        return self.forward(images, max_length)

    def forward(self, images, max_length=None):
        """Model-level seam (one reference mini-batch): logits (B, S, C) fp32, S = 101 with refinement, else the
        number of AR steps run; the repetition patch of parseq.py:301-309 is applied."""
        if max_length is not None:
            raise NotImplementedError("max_length is a training-time argument; inference uses None")
        h = self._ensure()
        x = images.detach().to(torch.float32).contiguous()
        B, _, Hh, W = x.shape
        if Hh != self.cfg.data.img_size[0]:
            raise ValueError("PARSeq expects height %d" % self.cfg.data.img_size[0])
        S, C = self.max_label_length + 1, self.num_classes
        logits = torch.zeros((B, S, C), dtype=torch.float32, device=x.device)
        ids = torch.empty((B, S), dtype=torch.int32)
        probs = torch.empty((B, S), dtype=torch.float32)
        rep = torch.empty((B,), dtype=torch.int32)
        steps = ctypes.c_int(0)
        _lib.check(_lib.lib().ytk_parseq_forward_f32(h, x.data_ptr(), 1 if x.is_cuda else 0, B, W, logits.data_ptr(),
                                                     1 if x.is_cuda else 0, ids.data_ptr(), probs.data_ptr(),
                                                     ctypes.byref(steps), rep.data_ptr(), None, None))
        if self._refine_iters == 0:
            logits = logits[:, : steps.value]
        if self.repetition_stop:
            for b, cut in enumerate(rep.tolist()):
                if cut >= 0 and cut < logits.shape[1]:
                    logits[b, cut, :] = -30.0
                    logits[b, cut, 0] = 30.0
        return logits

    def pack_crops(self, canvases, padded_widths, groups):
        """Packs canvases into one pinned uint8 buffer + ytk_crop descriptors (host side of recognize_crops)."""
        n = len(canvases)
        ph, pw = self.cfg.encoder.patch_size
        gh = self.cfg.data.img_size[0] // ph
        sizes = [int(c.shape[0] * c.shape[1] * 3) for c in canvases]
        total = int(sum(sizes))
        buf = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=torch.cuda.is_available())
        nb = buf.numpy()
        descs = (_lib.YtkCrop * max(n, 1))()
        off = tok = 0
        for i, c in enumerate(canvases):
            nb[off:off + sizes[i]] = np.ascontiguousarray(c).reshape(-1)
            wp = int(padded_widths[i])
            ntok = gh * (wp // pw)
            descs[i] = _lib.YtkCrop(off, int(c.shape[1]), wp, tok, ntok, int(groups[i]))
            off += sizes[i]
            tok += ntok
        return buf, total, descs, tok

    def run_packed(self, buf, total, descs, n, n_groups, stream=None):
        """Device call on a packed crop buffer (torch uint8 tensor, pinned host or cuda)."""
        h = self._ensure()
        S = self.max_label_length + 1
        ids = np.empty((n, S), dtype=np.int32)
        probs = np.empty((n, S), dtype=np.float32)
        glen = np.empty((max(n_groups, 1),), dtype=np.int32)
        _lib.check(_lib.lib().ytk_parseq_forward_crops(h, buf.data_ptr(), 1 if buf.is_cuda else 0, total, descs, n,
                                                       n_groups, ids.ctypes.data, probs.ctypes.data, glen.ctypes.data,
                                                       _stream_ptr(stream)))
        return ids, probs, glen[:n_groups]

    def run_packed_ptr(self, ptr, on_device, total, descs, n, n_groups, stream=None):
        """Device call on `total` bytes of crop canvases at address `ptr` (page-locked host or device memory); descs is
        a numpy structured array with the layout of ytk_crop."""
        h = self._ensure()
        S = self.max_label_length + 1
        ids = np.empty((n, S), dtype=np.int32)
        probs = np.empty((n, S), dtype=np.float32)
        glen = np.empty((max(n_groups, 1),), dtype=np.int32)
        dp = ctypes.cast(descs.ctypes.data, ctypes.POINTER(_lib.YtkCrop))
        _lib.check(_lib.lib().ytk_parseq_forward_crops(h, ptr, on_device, total, dp, n, n_groups, ids.ctypes.data,
                                                       probs.ctypes.data, glen.ctypes.data, _stream_ptr(stream)))
        return ids, probs, glen[:n_groups]

    def recognize_crops(self, canvases, padded_widths, groups, n_groups):
        """Fused ragged path.  canvases: list of (32, w_i, 3) uint8 RGB arrays (the reference's dataset.data[i]);
        padded_widths[i]: width the reference collate would pad crop i to; groups[i]: its mini-batch index.
        Returns ids (n,S) int32, probs (n,S) float32, group_len (n_groups,) int32 (numpy)."""
        buf, total, descs, _ = self.pack_crops(canvases, padded_widths, groups)
        return self.run_packed(buf, total, descs, len(canvases), n_groups)

    def last_flops(self):
        return _lib.lib().ytk_parseq_last_flops(self._ensure())

    def last_phase_ms(self):
        """CUDA-event times of the last forward: dict(encoder, ar, refine, copy) in ms."""
        a = (ctypes.c_float * 4)()
        _lib.lib().ytk_parseq_last_phase_ms(self._ensure(), a)
        return dict(zip(("encoder", "ar", "refine", "copy"), [float(v) for v in a]))


# ======================================================================================================== RT-DETRv2
def _rtdetr_anchors(img=640, strides=(8, 16, 32), grid_size=0.05, eps=1e-2):
    """`decoder.anchors` / `decoder.valid_mask` buffers of the reference (rtdetrv2_decoder.py:648-678): cell centres and
    level-scaled sizes in logit space, inf where any coordinate leaves (eps, 1 - eps)."""
    out = []
    for lvl, s in enumerate(strides):
        n = int(img / s)
        gy, gx = torch.meshgrid(torch.arange(n), torch.arange(n), indexing="ij")
        xy = (torch.stack([gx, gy], -1).unsqueeze(0) + 0.5) / torch.tensor([n, n], dtype=torch.float32)
        out.append(torch.cat([xy, torch.ones_like(xy) * grid_size * (2.0 ** lvl)], -1).reshape(-1, n * n, 4))
    a = torch.cat(out, 1)
    valid = ((a > eps) * (a < 1 - eps)).all(-1, keepdim=True)
    return torch.where(valid, torch.log(a / (1 - a)), torch.inf), valid


def _rtdetr_random_state_dict(num_classes, seed=0, img=640):
    """Random init with the reference's key set and shapes (RTDETRv2(cfg).state_dict(), from_pretrained=False) for an
    img x img input: the anchor buffers depend on it."""
    g = torch.Generator().manual_seed(seed)
    sd = OrderedDict()
    D, F, L, P, H = 256, 1024, 6, 12, 8

    def conv_norm(p, cout, cin, k, tracked):
        sd[p + ".conv.weight"] = _he_conv(g, cout, cin, k, k)
        sd[p + ".norm.weight"] = torch.ones(cout)
        sd[p + ".norm.bias"] = torch.zeros(cout)
        sd[p + ".norm.running_mean"] = torch.zeros(cout)
        sd[p + ".norm.running_var"] = torch.ones(cout)
        if tracked:
            sd[p + ".norm.num_batches_tracked"] = torch.tensor(0)

    def linear(p, cout, cin, bias=0.0):
        bound = math.sqrt(6.0 / (cin + cout))
        sd[p + ".weight"] = (torch.rand(cout, cin, generator=g) * 2 - 1) * bound
        sd[p + ".bias"] = torch.full((cout,), float(bias))

    def ln(p):
        sd[p + ".weight"] = torch.ones(D)
        sd[p + ".bias"] = torch.zeros(D)

    def mha(p):
        sd[p + ".in_proj_weight"] = (torch.rand(3 * D, D, generator=g) * 2 - 1) * math.sqrt(6.0 / (4 * D))
        sd[p + ".in_proj_bias"] = torch.zeros(3 * D)
        linear(p + ".out_proj", D, D)

    conv_norm("backbone.conv1.conv1_1", 32, 3, 3, False)
    conv_norm("backbone.conv1.conv1_2", 32, 32, 3, False)
    conv_norm("backbone.conv1.conv1_3", 64, 32, 3, False)
    cin = 64
    for s, (n, ch) in enumerate(zip((3, 4, 6, 3), (64, 128, 256, 512))):
        for b in range(n):
            p = "backbone.res_layers.%d.blocks.%d" % (s, b)
            conv_norm(p + ".branch2a", ch, cin, 1, False)
            conv_norm(p + ".branch2b", ch, ch, 3, False)
            conv_norm(p + ".branch2c", ch * 4, ch, 1, False)
            if b == 0:
                conv_norm(p + (".short.conv" if s else ".short"), ch * 4, cin, 1, False)
            cin = ch * 4
    for i, c in enumerate((512, 1024, 2048)):
        conv_norm("encoder.input_proj.%d" % i, D, c, 1, True)
    p = "encoder.encoder.0.layers.0"
    mha(p + ".self_attn")
    linear(p + ".linear1", F, D)
    linear(p + ".linear2", D, F)
    ln(p + ".norm1")
    ln(p + ".norm2")
    for kind in ("fpn_blocks", "pan_blocks"):
        for i in range(2):
            q = "encoder.%s.%d" % (kind, i)
            conv_norm(q + ".conv1", D, 2 * D, 1, True)
            conv_norm(q + ".conv2", D, 2 * D, 1, True)
            for j in range(3):
                conv_norm("%s.bottlenecks.%d.conv1" % (q, j), D, D, 3, True)
                conv_norm("%s.bottlenecks.%d.conv2" % (q, j), D, D, 1, True)
    for i in range(2):
        conv_norm("encoder.lateral_convs.%d" % i, D, D, 1, True)
        conv_norm("encoder.downsample_convs.%d" % i, D, D, 3, True)
    sd["decoder.anchors"], sd["decoder.valid_mask"] = _rtdetr_anchors(img)
    for i in range(3):
        conv_norm("decoder.input_proj.%d" % i, D, D, 1, True)
    prior = -math.log(99.0)
    for i in range(L):
        p = "decoder.decoder.layers.%d" % i
        mha(p + ".self_attn")
        ln(p + ".norm1")
        sd[p + ".cross_attn.num_points_scale"] = torch.full((P,), 0.25)
        sd[p + ".cross_attn.sampling_offsets.weight"] = torch.zeros(H * P * 2, D)
        th = torch.arange(H, dtype=torch.float32) * (2.0 * math.pi / H)
        gi = torch.stack([th.cos(), th.sin()], -1)
        gi = (gi / gi.abs().max(-1, keepdim=True).values).reshape(H, 1, 2).tile([1, P, 1])
        sd[p + ".cross_attn.sampling_offsets.bias"] = (gi * torch.arange(1, 5).repeat(3).reshape(1, -1, 1)).flatten()
        sd[p + ".cross_attn.attention_weights.weight"] = torch.zeros(H * P, D)
        sd[p + ".cross_attn.attention_weights.bias"] = torch.zeros(H * P)
        linear(p + ".cross_attn.value_proj", D, D)
        linear(p + ".cross_attn.output_proj", D, D)
        ln(p + ".norm2")
        linear(p + ".linear1", F, D)
        linear(p + ".linear2", D, F)
        ln(p + ".norm3")
        linear("decoder.dec_score_head.%d" % i, num_classes, D, prior)
        for j, (co, ci) in enumerate(((D, D), (D, D), (4, D))):
            linear("decoder.dec_bbox_head.%d.layers.%d" % (i, j), co, ci)
        sd["decoder.dec_bbox_head.%d.layers.2.weight" % i].zero_()
    sd["decoder.denoising_class_embed.weight"] = torch.randn(num_classes + 1, D, generator=g)
    linear("decoder.query_pos_head.layers.0", 2 * D, 4)
    linear("decoder.query_pos_head.layers.1", D, 2 * D)
    linear("decoder.enc_output.proj", D, D)
    ln("decoder.enc_output.norm")
    linear("decoder.enc_score_head", num_classes, D, prior)
    for j, (co, ci) in enumerate(((D, D), (D, D), (4, D))):
        linear("decoder.enc_bbox_head.layers.%d" % j, co, ci)
    sd["decoder.enc_bbox_head.layers.2.weight"].zero_()
    return sd


class RTDETRv2(_DeviceModel):
    """reference models/rtdetr.py:9-22 (PResNet-50d + HybridEncoder + RTDETRTransformerv2, eval).  `model(tensor)` takes
    the (n, 3, S, S) fp32 tensor in [0, 1] that LayoutParser / TableStructureRecognizer / CellDetector.preprocess produce
    (S = cfg.data.img_size: 640, 960 for the cell detector) and returns {"pred_logits": (n, Q, C), "pred_boxes": (n, Q, 4)}
    (Q = num_queries: 300, 1500 for the cell detector) on the tensor's device.  The forward is the sm_100a engine
    behind ytk_rtdetr_forward_f32 (csrc/rtdetr_engine.cu); there is no CPU fallback."""

    def __init__(self, cfg=None, seed=0):
        super().__init__()
        self.cfg = cfg
        d = cfg.RTDETRTransformerv2 if cfg is not None else None
        self.num_classes = int(d.num_classes) if d is not None else 6
        self.num_queries = int(d.num_queries) if d is not None else 300
        self.img_size = int(cfg.data.img_size[0]) if cfg is not None else 640
        if cfg is not None and (list(cfg.data.img_size) != [self.img_size] * 2 or
                                list(d.eval_spatial_size) != [self.img_size] * 2):
            raise ValueError("RTDETRv2: square img_size == eval_spatial_size expected, got %s / %s"
                             % (list(cfg.data.img_size), list(d.eval_spatial_size)))
        self._sd = _rtdetr_random_state_dict(self.num_classes, seed, self.img_size)

    def _ensure(self):
        self._require_cuda()
        if self._handle is None:
            tab, keep = _lib.tensor_table(self._sd)
            h = ctypes.c_void_p()
            with torch.cuda.device(self.cuda_device()):
                _lib.check(_lib.lib().ytk_rtdetr_create(tab, len(tab), self.num_classes, self.num_queries, self.img_size,
                                                        ctypes.byref(h)))
            self._handle = h
        return self._handle

    def _release(self):
        if self._handle is not None:
            _lib.lib().ytk_rtdetr_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    def __call__(self, tensor, targets=None):
        return self.forward(tensor)

    def forward(self, tensor, stream=None):
        h = self._ensure()
        S = self.img_size
        if tensor.dim() != 4 or tuple(tensor.shape[1:]) != (3, S, S):
            raise ValueError("RTDETRv2 expects (n, 3, %d, %d), got %s" % (S, S, tuple(tensor.shape)))
        x = tensor.detach().to(torch.float32).contiguous()
        n = x.shape[0]
        logits = torch.empty((n, self.num_queries, self.num_classes), dtype=torch.float32, device=x.device)
        boxes = torch.empty((n, self.num_queries, 4), dtype=torch.float32, device=x.device)
        on_dev = 1 if x.is_cuda else 0
        _lib.check(_lib.lib().ytk_rtdetr_forward_f32(h, x.data_ptr(), on_dev, n, logits.data_ptr(), boxes.data_ptr(), on_dev,
                                                     _stream_ptr(stream)))
        return {"pred_logits": logits, "pred_boxes": boxes}

    def flops(self, n=1):
        return _lib.lib().ytk_rtdetr_flops(self._ensure(), n)

    def device_bytes(self, n=1):
        """Device bytes of the activation buffers of the batch-n engine."""
        return int(_lib.lib().ytk_rtdetr_device_bytes(self._ensure(), n))

    def debug_tensor(self, n, name):
        """Intermediate activation of the last forward of batch size n (test hook) as a numpy array."""
        cap = 64 << 20
        buf = torch.empty(cap, dtype=torch.float32)
        shape = (ctypes.c_int * 4)()
        _lib.check(_lib.lib().ytk_rtdetr_debug_tensor(self._ensure(), n, name.encode(), buf.data_ptr(), cap, shape))
        dims = [int(v) for v in shape]
        return buf[: dims[0] * dims[1] * dims[2] * dims[3]].reshape(dims).numpy().copy()
