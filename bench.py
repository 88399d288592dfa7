"""Benchmark of the DBNet -> PARSeq OCR hot path (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W               # this repo's CUDA path
    python bench.py ... --dump-outputs DIR                      # + the last timed step's outputs as DIR/*.npy
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                        # the reference's CPU implementation (oracle restatement)

One step = the hot path over one batch of synthetic 1200x1600 (H x W) pages per GPU (~200 text lines each):
DBNet (`dbnetv2_1`) on every page + PARSeq (`parseq-large-v4_1`, dynamic_width + batch_bucketing) on every crop.
  value : pages/s with the pages already resident in HBM (device time only, CUDA events): detector, crop kernels
          (ytk_extract_crops_u8) and recognizer; with more than one GPU the mini-batch groups are balanced across ranks
          inside the timed region (GPU-to-GPU all_to_all crop scatter + result gather, yomitoku_b200/parallel.py)
  e2e   : pages/s through the public batched API (`BatchedOCR.stream`) from HOST pages: H2D pages, DBNet, D2H of the
          probability maps, host post-processing (process pool; contours / unclip as the reference does on the host),
          crop records H2D, crop kernels, PARSeq, D2H ids/probs, tokenizer decode.  Random detector weights do not
          produce text boxes, so the host post-processor consumes a synthetic probability map of the page's
          ground-truth boxes (the detector still runs and its output still crosses PCIe), per SURVEY.md section 8d.
Multi-GPU default (`--skew auto`): even ranks hold pages with 280 text lines, odd ranks pages with 120 (same 200-line
mean and the same total work as the single-GPU run), so the crop scatter has to move groups; the line reports the
bytes it moved and the time it took.  Weights are seeded random (no checkpoints offline); with random PARSeq weights no
row emits EOS, so every AR loop runs all 101 steps (worst case) - `other_configs` adds a trained-like run that stops
early, BASELINE config 2 (one page through DBNet) and config 3 (512 crops through PARSeq).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pages/sec (DBNet->PARSeq OCR, synthetic 1600x1200 pages, ~200 crops/page)"
WORKLOAD = "OCR DBNet(dbnetv2_1)->PARSeq(parseq-large-v4_1), synthetic 1200x1600 pages, ~200 text lines/page"
PAGES_PER_GPU = 16
REC_MODEL = "parseq-large-v4_1"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0),
                "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [t.strip() for t in o.strip().split(",")]
                if len(f) >= 7:
                    self.rows.append(f)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------ CPU arm
_CPU_THREADS = None


def _pick_cpu_threads(det_sd, x):
    """Thread sweep on the detector forward (the largest fp32 eager kernels of the path): the reference's PyTorch CPU
    path is timed with the intra-op thread count that is fastest on this box, not an arbitrary cap."""
    global _CPU_THREADS
    if _CPU_THREADS is not None:
        return _CPU_THREADS
    from oracle import dbnet as odb
    ncpu = os.cpu_count() or 1
    # (more intra-op threads than 64 collapse on this workload: 128 threads took 26 s for the probe in round 2)
    cands = sorted({t for t in (8, 16, 32, 64) if t <= ncpu} | {min(ncpu, 8)})
    sweep = {}
    xs = x[:, :, :384, :512].contiguous()      # a quarter-size map is enough to rank the settings
    for t in cands:
        torch.set_num_threads(t)
        odb.dbnet_forward(det_sd, xs)
        t0 = time.perf_counter()
        odb.dbnet_forward(det_sd, xs)
        sweep[t] = time.perf_counter() - t0
    best = min(sweep, key=sweep.get)
    torch.set_num_threads(best)
    _CPU_THREADS = (best, {str(k): round(v, 3) for k, v in sweep.items()})
    return _CPU_THREADS


def cpu_page_rate(det_sd=None, rec_sd=None):
    """The reference's CPU implementation of the path (oracle restatement of its fp32 eager PyTorch modules) on ONE FULL
    page: DBNet + post-processing + all ~200 crops through PARSeq-large with the reference's own batching (sorted
    chunks of 128, dynamic width).  Nothing is extrapolated.  Returns a dict."""
    from oracle import dbnet as odb
    from oracle import parseq as ops
    from oracle import pipeline as opipe
    from yomitoku_b200.config import TextRecognizerPARSeqLargeV41Config, load_config
    from yomitoku_b200.models import _dbnet_random_state_dict, _parseq_random_state_dict
    from yomitoku_b200.synth import synthetic_page, synthetic_prob_map
    page, quads = synthetic_page(0)
    if det_sd is None:
        det_sd = _dbnet_random_state_dict(0)
    cfg = load_config(TextRecognizerPARSeqLargeV41Config)
    if rec_sd is None:
        rec_sd = _parseq_random_state_dict(cfg, 0)
    spec = ops.SPECS[REC_MODEL]
    tok = ops.Tokenizer(open(cfg.charset, encoding="utf-8").read())
    x = opipe.detector_preprocess(page)
    threads, sweep = _pick_cpu_threads(det_sd, x)
    t0 = time.perf_counter()
    x = opipe.detector_preprocess(page)
    odb.dbnet_forward(det_sd, x)
    t_det = time.perf_counter() - t0
    prob = synthetic_prob_map(quads, (1184, 1600), (1200, 1600))
    t0 = time.perf_counter()
    opipe.dbnet_postprocess(prob, (1200, 1600))
    t_post = time.perf_counter() - t0
    t0 = time.perf_counter()
    opipe.recognize(rec_sd, spec, tok, page, quads, dynamic_width=True, batch_bucketing=True, batch_size=128)
    t_rec = time.perf_counter() - t0
    per_page = t_det + t_post + t_rec
    return {"pages_per_s": 1.0 / per_page, "t_det_s": t_det, "t_post_s": t_post, "t_rec_s": t_rec,
            "crops": len(quads), "cores": threads, "thread_sweep_s": sweep, "host_cores": os.cpu_count()}


def _cpu_sample_text(r):
    return ("one FULL page, nothing extrapolated: DBNet fp32 (%.2f s) + post-processing (%.3f s) + all %d crops through "
            "PARSeq %s with the reference's batching of 128 (%.2f s); oracle = restated reference fp32 eager path; "
            "intra-op threads %d of %d host cores chosen by a sweep on the detector forward %s"
            % (r["t_det_s"], r["t_post_s"], r["crops"], REC_MODEL, r["t_rec_s"], r["cores"], r["host_cores"],
               json.dumps(r["thread_sweep_s"])))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, detail = [], None
    t_start = time.perf_counter()
    warm, steps, i = min(args.warmup, 1), args.steps, 0
    while i < warm + steps:
        r = cpu_page_rate()
        if i >= warm:
            vals.append(r["pages_per_s"])
            detail = r
        i += 1
        per = (time.perf_counter() - t_start) / i
        if per * (warm + steps) > 200.0:       # keep the whole run within a few minutes (a step = one full page)
            steps = max(1, int(200.0 / per) - warm)
    if not vals:
        vals, detail = [r["pages_per_s"]], r
    v = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "pages/s", "n_gpus": args.gpus, "steps": len(vals),
        "warmup": warm, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "note": "reference CPU path = oracle restatement of yomitoku's PyTorch fp32 eager modules; one step = "
                           "one full page (DBNet + post-processing + ~200 crops, reference batching)"},
        "cpu_baseline": {"value": v, "unit": "pages/s", "cores": detail["cores"], "kind": "port",
                         "sample": _cpu_sample_text(detail)},
        "e2e": {"value": v, "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm helpers
DUMP_PROB_VALUES = 1 << 22      # probability-map values kept by --dump-outputs (16 MB of ~120 MB per step)


def dump_outputs(out_dir, prefix, prob_dev, post, rec_out):
    """--dump-outputs: what the last timed step handed its caller, as out_dir/<prefix><name>.npy (float32 / float64,
    ~20 MB with the default --pages), so that two builds can be compared output for output on identical inputs:
      det_prob_sample        the detector's probability maps (pages, H, W), values at DUMP_PROB_VALUES fixed positions
                             (ascending flat indices drawn with numpy seed 0)
      post_meta              (pages, 4) of the device post-processing front: runs, components, 4 x Euler number, overflow
      post_runs              (n, 6) = page, root, y, x0, x1, sum of every row run of the last detector batch's pages,
                             sorted by (page, y, x0)
      rec_ids, rec_probs     (crops, S) token ids / probabilities of every crop, mini-batch groups in bench order
      rec_group_steps        (groups,) decode steps of every mini-batch group
    `post` = (meta, runs, first page of the last detector batch) or None when the front did not run."""
    from yomitoku_b200.models import DB_RUN_DTYPE
    os.makedirs(out_dir, exist_ok=True)
    flat = prob_dev.reshape(-1)
    n = flat.numel()
    if n > DUMP_PROB_VALUES:
        idx = np.sort(np.random.default_rng(0).choice(n, DUMP_PROB_VALUES, replace=False))
        flat = flat[torch.from_numpy(idx).to(flat.device)]
    arrays = {"det_prob_sample": flat.cpu().numpy().astype(np.float32)}
    if post is not None:
        meta, runs, first = post
        meta = meta.cpu().numpy()
        runs = runs.cpu().numpy()
        rows = []
        for j in range(meta.shape[0] - first):
            r = runs[j].reshape(-1).view(DB_RUN_DTYPE)[:min(int(meta[first + j, 0]), runs.shape[1])]
            rows.append(np.stack([np.full(len(r), first + j, np.float64)] +
                                 [r[f].astype(np.float64) for f in ("root", "y", "x0", "x1", "sum")], axis=1))
        rows = np.concatenate(rows)
        arrays["post_meta"] = meta.astype(np.float64)
        arrays["post_runs"] = rows[np.lexsort((rows[:, 3], rows[:, 2], rows[:, 0]))]
    arrays["rec_ids"] = np.concatenate([ids for ids, _, _ in rec_out]).astype(np.float32)
    arrays["rec_probs"] = np.concatenate([probs for _, probs, _ in rec_out]).astype(np.float32)
    arrays["rec_group_steps"] = np.array([glen for _, _, glen in rec_out], np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, prefix + name + ".npy"), a)
    print("[bench] outputs of the last timed step: %s (%.1f MB)" % (
        ", ".join("%s%s %s" % (prefix, k, tuple(a.shape)) for k, a in arrays.items()),
        sum(a.nbytes for a in arrays.values()) / 2**20), file=sys.stderr, flush=True)


def _gemm_window(L, fn):
    from yomitoku_b200 import _lib
    f, ms, n = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_longlong(0)
    L.ytk_gemm_profile_begin()
    fn()
    torch.cuda.synchronize()
    _lib.check(L.ytk_gemm_profile_end(ctypes.byref(f), ctypes.byref(ms), ctypes.byref(n)))
    return {"tflop": f.value / 1e12, "ms": ms.value, "launches": int(n.value),
            "achieved": f.value / 1e12 / (ms.value / 1e3) if ms.value > 0 else 0.0}


def _time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def config2_line(det, L, pk, steps=20, warmup=5):
    """BASELINE config 2: TextDetector DBNet, ONE synthetic 1600x1200 page, 1 B200 - latency of the device path (page
    resident in HBM -> probability map in HBM) and its tensor roofline."""
    from yomitoku_b200 import _lib
    from yomitoku_b200.synth import synthetic_page
    page, _ = synthetic_page(0)
    Hn, Wn = det.model.input_size(1200, 1600)
    pd = torch.from_numpy(page)[None].cuda()
    out = torch.empty((1, Hn, Wn), dtype=torch.float32, device="cuda")

    def step():
        _lib.check(L.ytk_dbnet_forward_u8(det.model._ensure(), pd.data_ptr(), 1, 1, 1200, 1600, out.data_ptr(), 1, None))
    ms = _time_ms(step, steps, warmup)
    flops = det.model.flops(1, Hn, Wn)
    g = _gemm_window(L, step)
    return {"metric": "pages/sec (DBNet TextDetector, one 1600x1200 page, batch 1)", "value": 1e3 / ms, "unit": "pages/s",
            "ms_per_step": ms, "steps": steps, "warmup": warmup, "dtype": "f16", "higher_is_better": True,
            "config": {"workload": "BASELINE config 2: TextDetector DBNet(dbnetv2_1), single synthetic 1200x1600 page, "
                                   "1 B200, page and probability map resident in HBM, batch 1 (latency)"},
            "roofline": {"bound": "tensor", "achieved": flops / 1e12 / (ms / 1e3), "peak": pk["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": flops / 1e12 / (ms / 1e3) / pk["bf16_tflops"],
                         "gflop_per_page": flops / 1e9, "peak_source": pk["source"] + " bf16_tflops (burst: short run)",
                         "gemm_kernel": g}}


def config5_layout_line(L, pk, batch=8, steps=10, warmup=3):
    """The model BASELINE config 5 adds to the OCR path: RT-DETRv2 (layout parser; the table structure recognizer is the
    same network with 3 classes), `batch` synthetic 640x640 inputs resident in HBM -> pred_logits / pred_boxes in HBM."""
    from yomitoku_b200 import _lib
    from yomitoku_b200.config import LayoutParserRTDETRv2V2Config, to_config
    from yomitoku_b200.models import RTDETRv2
    m = RTDETRv2(cfg=to_config(LayoutParserRTDETRv2V2Config())).to("cuda")
    x = torch.rand(batch, 3, 640, 640, device="cuda")
    lg = torch.empty((batch, 300, 6), dtype=torch.float32, device="cuda")
    bx = torch.empty((batch, 300, 4), dtype=torch.float32, device="cuda")

    def step():
        _lib.check(L.ytk_rtdetr_forward_f32(m._ensure(), x.data_ptr(), 1, batch, lg.data_ptr(), bx.data_ptr(), 1, None))
    ms = _time_ms(step, steps, warmup)
    flops = m.flops(batch)
    g = _gemm_window(L, step)
    return {"metric": "images/sec (RT-DETRv2 layout parser forward, 640x640, batch %d)" % batch,
            "value": batch / (ms / 1e3), "unit": "images/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
            "dtype": "f16", "higher_is_better": True,
            "config": {"workload": "BASELINE config 5's extra model: RT-DETRv2 (PResNet-50d + HybridEncoder + 6-layer "
                                   "deformable decoder, 300 queries), %d synthetic 640x640 inputs, 1 B200, inputs and outputs "
                                   "resident in HBM, random weights" % batch},
            "roofline": {"bound": "tensor", "achieved": flops / 1e12 / (ms / 1e3), "peak": pk["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": flops / 1e12 / (ms / 1e3) / pk["bf16_tflops"],
                         "gflop_per_image": flops / batch / 1e9, "peak_source": pk["source"] + " bf16_tflops (burst: short run)",
                         "gemm_kernel": g}}


def config3_line(rec, L, pk, n_crops=512, steps=5, warmup=3):
    """BASELINE config 3: TextRecognizer PARSeq (full), 512 crops, dynamic_width + batch_bucketing, 1 B200: crops/s with
    the crops resident in HBM (reference grouping: sorted chunks of 128, each padded to its own maximum)."""
    from yomitoku_b200.data import ParseqDataset
    from yomitoku_b200.synth import synthetic_page
    from yomitoku_b200.text_recognizer import plan_mini_batches
    canv, cw = [], []
    pi = 100
    while len(canv) < n_crops:
        pg, q = synthetic_page(pi)
        ds = ParseqDataset(rec._cfg, pg, q, dynamic_width=True)
        canv += ds.data
        cw += ds.content_widths
        pi += 1
    canv, cw = canv[:n_crops], cw[:n_crops]
    order = np.argsort(cw).tolist()
    plan = plan_mini_batches([c.shape[1] for c in canv], order, True, rec._cfg.data.batch_size, None, None)
    padded, group = rec._collate_widths(canv, plan)
    fc = [canv[i] for b in plan for i in b]
    fp = [padded[i] for b in plan for i in b]
    fg = [group[i] for b in plan for i in b]
    buf, total, descs, n_tok = rec.model.pack_crops(fc, fp, fg)
    bd = buf.cuda()

    def step():
        rec.model.run_packed(bd, total, descs, n_crops, len(plan))
    ms = _time_ms(step, steps, warmup)
    flops = rec.model.last_flops()
    return {"metric": "crops/sec (PARSeq TextRecognizer, 512 crops, dynamic_width + batch_bucketing)",
            "value": n_crops / (ms / 1e3), "unit": "crops/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
            "dtype": "f16", "higher_is_better": True,
            "config": {"workload": "BASELINE config 3: TextRecognizer PARSeq(%s), 512 synthetic crops, dynamic_width + "
                                   "batch_bucketing, 1 B200, crops resident in HBM; %d mini-batches, %d encoder tokens, "
                                   "101 AR steps (random weights)" % (REC_MODEL, len(plan), n_tok),
                       "recognizer_phase_ms": rec.model.last_phase_ms()},
            "roofline": {"bound": "tensor", "achieved": flops / 1e12 / (ms / 1e3), "peak": pk["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": flops / 1e12 / (ms / 1e3) / pk["bf16_tflops"],
                         "gflop_per_step": flops / 1e9, "peak_source": pk["source"] + " bf16_tflops (burst: short run)"}}


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pages", type=int, default=PAGES_PER_GPU, help="pages per GPU per step")
    ap.add_argument("--skew", default="auto", choices=["auto", "0", "1"],
                    help="per-rank line-count skew (280 / 120 lines on even / odd ranks); auto = on with > 1 GPU")
    ap.add_argument("--weights", default="random", choices=["random", "peaked"],
                    help="peaked: trained-like PARSeq weights whose rows emit EOS (AR loop stops early)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip other_configs (config 2, config 3, EOS run)")
    ap.add_argument("--no-window", action="store_true", help="skip the instrumented per-launch GEMM timing step "
                                                               "(for runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from yomitoku_b200 import TextDetector, TextRecognizer, _lib
    from yomitoku_b200 import parallel as par
    from yomitoku_b200.data import crop_geometry
    from yomitoku_b200.models import extract_crops_device
    from yomitoku_b200.pipeline import BatchedOCR, _PageGeoms
    from yomitoku_b200.synth import peaked_parseq_state_dict, synthetic_page, synthetic_prob_map
    from yomitoku_b200.text_recognizer import plan_mini_batches

    det = TextDetector(from_pretrained=False, device="cuda")
    rec = TextRecognizer(model_name=REC_MODEL, from_pretrained=False, device="cuda", dynamic_width=True,
                         batch_bucketing=True)
    if args.weights == "peaked":
        rec.model.load_state_dict(peaked_parseq_state_dict(rec.model.state_dict()))
    if world > 1:
        # one-time weight broadcast from rank 0 over NCCL (all ranks then hold identical weights)
        det.model.load_state_dict(par.broadcast_state_dict(det.model.state_dict(), "cuda"))
        rec.model.load_state_dict(par.broadcast_state_dict(rec.model.state_dict(), "cuda"))
    L = _lib.lib()
    P = args.pages
    skew = (world > 1) if args.skew == "auto" else (args.skew == "1")
    n_slots = (7 if rank % 2 == 0 else 3) if skew else 5
    pages, quads = [], []
    for i in range(P):
        pg, q = synthetic_page(rank * P + i, n_slots=n_slots)
        pages.append(pg)
        quads.append(q)
    Hn, Wn = det.model.input_size(1200, 1600)
    probs_syn = [synthetic_prob_map(q, (Hn, Wn), (1200, 1600)) for q in quads]
    ncpu = os.cpu_count() or 2
    ocr = BatchedOCR(det, rec, det_batch=8, workers=max(2, min(32, (ncpu - 2 * world) // world)), device_crops=True)
    # ---------------- device-resident inputs for `value`
    pages_dev = torch.from_numpy(np.stack(pages)).cuda()
    prob_dev = torch.empty((P, Hn, Wn), dtype=torch.float32, device="cuda")

    # device front half of the post-processing (threshold, components, row runs): it runs on the synthetic maps, the
    # random-weight maps above are noise
    syn_dev = torch.from_numpy(np.stack(probs_syn)).cuda()
    post_labels = torch.empty((ocr.det_batch, Hn, Wn), dtype=torch.int32, device="cuda")
    post_runs = torch.empty((ocr.det_batch, 32768, 24), dtype=torch.uint8, device="cuda")
    post_meta = torch.empty((P, 4), dtype=torch.int32, device="cuda")

    def det_step():
        for s in range(0, P, ocr.det_batch):
            e = min(P, s + ocr.det_batch)
            _lib.check(L.ytk_dbnet_forward_u8(det.model._ensure(), pages_dev[s:e].data_ptr(), 1, e - s, 1200, 1600,
                                              prob_dev[s:e].data_ptr(), 1, None))
            if det.device_post:
                _lib.check(L.ytk_dbnet_post_front(syn_dev[s:e].data_ptr(), e - s, Hn, Wn, float(det.post_processor.thresh), post_labels.data_ptr(),
                                                  post_labels.numel() * 4, post_runs.data_ptr(), 32768,
                                                  post_meta[s:e].data_ptr(), None))

    # per-page crop records + reference grouping (exactly what BatchedOCR.recognize_pooled builds from the host stage)
    per_page, base = [], 0
    for pi, q in enumerate(quads):
        g, keep = crop_geometry((1200, 1600), q, rec._cfg.data.img_size, True, page=pi)
        per_page.append((_PageGeoms(g, base), g["cw"].tolist(), len(q)))
        base += len(g)
    geoms_all = np.concatenate([p[0].geoms for p in per_page])
    groups = []
    for canv, cw, nq in per_page:
        order = np.argsort(cw).tolist()
        plan = plan_mini_batches(canv.widths, order, True, rec._cfg.data.batch_size, None, None)
        padded, _ = rec._collate_widths(canv.widths, plan)
        for b in plan:
            groups.append(([canv.widths[i] for i in b], [padded[i] for i in b], canv.base + np.asarray(b, np.int64)))
    n_crops = len(geoms_all)
    if rank == 0 and world == 1:
        # the device-cut canvases are the reference's canvases, bit for bit (one page checked here, all in the tests)
        from yomitoku_b200.data import ParseqDataset
        ds = ParseqDataset(rec._cfg, pages[0], quads[0], dynamic_width=True)
        g0 = np.ascontiguousarray(per_page[0][0].geoms)
        chk, chk_total = extract_crops_device(pages_dev, g0)
        if not np.array_equal(chk.cpu().numpy()[:chk_total], np.concatenate([c.reshape(-1) for c in ds.data])):
            raise RuntimeError("device-cut canvases differ from the OpenCV canvases")
        del chk

    # the host-side plan of the packed call (chunks, records, descriptors) is input preparation, like the resident pages
    plan = ocr._plan_groups_dev(groups, geoms_all) if world == 1 else None

    def rec_step():
        # single GPU: everything stays local; several GPUs: cost gather, balancing, GPU-to-GPU crop scatter, recognition
        # of own + received groups, result gather - all inside the timed region
        return ocr._run_groups_dev(groups, geoms_all, pages_dev, None, None, plan)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        det_step()
        rec_step()
    sync_all()
    launches0 = L.ytk_launch_count()
    x0 = dict(par.STATS)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    det_ms = rec_ms = 0.0
    with ClockSampler(local) as clocks:
        t_all0 = torch.cuda.Event(enable_timing=True)
        t_all1 = torch.cuda.Event(enable_timing=True)
        t_all0.record()
        for _ in range(args.steps):
            ev[0].record()
            det_step()
            ev[1].record()
            rec_out = rec_step()
            ev[2].record()
            torch.cuda.synchronize()
            det_ms += ev[0].elapsed_time(ev[1])
            rec_ms += ev[1].elapsed_time(ev[2])
        t_all1.record()
        sync_all()
        total_ms = t_all0.elapsed_time(t_all1)
    launches = L.ytk_launch_count() - launches0
    x_value = {k: par.STATS[k] - x0[k] for k in x0}
    ar_steps = int(L.ytk_parseq_last_steps(rec.model._ensure()))
    phase_value = rec.model.last_phase_ms()     # CUDA-event phase times of the last recognizer call of the timed region
    rec_flops_local = rec.model.last_flops()
    if args.dump_outputs:
        post = (post_meta, post_runs, (P - 1) // ocr.det_batch * ocr.det_batch) if det.device_post else None
        dump_outputs(args.dump_outputs, "rank%d_" % rank if world > 1 else "", prob_dev, post, rec_out)
    tm = torch.tensor([total_ms, det_ms, rec_ms], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([float(n_crops), float(x_value["exchange_bytes_sent"]), float(x_value["exchange_ms"]),
                        rec_flops_local], dtype=torch.float64, device="cuda")
    cmax = cnt.clone()
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        dist.all_reduce(cmax, op=dist.ReduceOp.MAX)
    total_ms, det_ms, rec_ms = [float(v) for v in tm.tolist()]
    crops_all, xbytes_all, _, rec_flops_all = [float(v) for v in cnt.tolist()]
    value = world * P * args.steps / (total_ms / 1e3)
    det_flops = det.model.flops(ocr.det_batch, Hn, Wn) / ocr.det_batch * P
    pk = peaks()
    det_tflops = det_flops * args.steps / (det_ms / 1e3) / 1e12
    rec_tflops = rec_flops_all / world * args.steps / (rec_ms / 1e3) / 1e12   # per-GPU average over the slowest rank's time
    # ---------------- per-launch timing of the dominant kernel (one instrumented extra step, outside the timed region)
    if args.no_window:
        g_det = g_rec = {"tflop": 0.0, "ms": 1e-9, "launches": 0, "achieved": 0.0}
    else:
        g_det = _gemm_window(L, det_step)
        g_rec = _gemm_window(L, rec_step)
    # ---------------- e2e through the public batched API from host pages
    e2e = None
    if not args.no_e2e:
        nw = max(3, args.warmup)
        # the synthetic maps stand in for the detector's output (random weights give noise): with the device-side
        # post-processing that output lives in HBM, so the stand-ins are device tensors too (a D2D copy per page)
        po = [torch.from_numpy(p).cuda() for p in probs_syn] if det.device_post else probs_syn
        for _ in ocr.stream([pages] * nw, lookahead=2, prob_override=[po] * nw):
            pass
        sync_all()
        x1 = dict(par.STATS)
        d2h0, front0, host0 = ocr.post_d2h_bytes, ocr.post_front_pages, ocr.post_host_pages
        t0 = time.perf_counter()
        n_words = 0
        # documented pipelined use of the public API: `BatchedOCR.stream` runs the detector + host stage of the next
        # batches (own thread, own CUDA stream, process pool) while the recognizer works on the current one; exactly
        # `steps` batches of P pages go through
        for res in ocr.stream([pages] * args.steps, lookahead=2, prob_override=[po] * args.steps):
            n_words += sum(len(r.words) for r in res)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        x_e2e = {k: par.STATS[k] - x1[k] for k in x1}
        tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
        xs = torch.tensor([float(x_e2e["exchange_bytes_sent"]), float(n_words)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(xs, op=dist.ReduceOp.SUM)
        dt = float(tt.item())
        # the crops never cross PCIe, only their 136-byte records do; results: ids + probs per crop; detector stage:
        # the components' row runs (24 bytes each) instead of the maps when the device post-processing front runs
        h2d = P * 1200 * 1600 * 3 + n_crops * 136
        d2h = (ocr.post_d2h_bytes - d2h0) // args.steps + n_crops * 101 * 8
        e2e = {"value": world * P * args.steps / dt, "unit": "pages/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "words_per_page": float(xs[1].item()) / (args.steps * P * world),
               "host_workers": ocr.workers, "device_crops": True, "device_post": bool(det.device_post),
               "post_front_pages": ocr.post_front_pages - front0, "post_host_fallback_pages": ocr.post_host_pages - host0,
               "exchange_bytes_per_step_all_ranks": float(xs[0].item()) / args.steps,
               "exchange_ms_per_step_rank0": x_e2e["exchange_ms"] / args.steps}
    # ---------------- other configs (single GPU only: they are single-GPU configurations of BASELINE.json)
    other = []
    if world == 1 and not args.no_extra:
        other.append(config2_line(det, L, pk))
        other.append(config3_line(rec, L, pk))
        other.append(config5_layout_line(L, pk))
        if args.weights == "random":
            # the same step with trained-like weights whose rows emit EOS: the AR loop stops when every row of a
            # mini-batch holds an EOS, which shifts the step towards the encoder
            sd_random = rec.model.state_dict()
            rec.model.load_state_dict(peaked_parseq_state_dict(sd_random))
            ms = _time_ms(lambda: (det_step(), rec_step()), 3, 2)
            ph = rec.model.last_phase_ms()
            other.append({"metric": METRIC, "value": P / (ms / 1e3), "unit": "pages/s", "ms_per_step": ms, "steps": 3,
                          "warmup": 2, "dtype": "f16", "higher_is_better": True,
                          "config": {"workload": WORKLOAD + "; trained-LIKE PARSeq weights (synth.peaked_parseq_state_dict): "
                                                 "rows emit EOS, AR loop stops early",
                                     "ar_steps_last_call": int(L.ytk_parseq_last_steps(rec.model._ensure())),
                                     "recognizer_phase_ms": ph}})
            rec.model.load_state_dict(sd_random)
    ocr.close()
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_page_rate(det.model.state_dict(), rec.model.state_dict())
        cpu = {"value": r["pages_per_s"], "unit": "pages/s", "cores": r["cores"], "kind": "port",
               "sample": _cpu_sample_text(r)}
    if rank == 0:
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "r02_bench_step_traffic.json")
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic, traffic_src = tj["gemm_tc_kernel_dram_bytes_per_step"], tj.get("source")
            except Exception:
                pass
        g_ms = g_det["ms"] + g_rec["ms"]
        g_tf = g_det["tflop"] + g_rec["tflop"]
        line = {
            "metric": METRIC, "value": value, "unit": "pages/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "pages_per_gpu_per_step": P, "crops_per_step_all_ranks": int(crops_all),
                       "parallelism": "pages sharded %d/GPU for detection; recognition: reference mini-batch groups "
                                      "balanced across ranks (GPU-to-GPU all_to_all crop scatter + result gather) in both "
                                      "value and e2e" % P,
                       "skew": ("even ranks 280 text lines/page, odd ranks 120 (mean 200)" if skew else
                                "none: 200 text lines on every page"),
                       "l2": "working set (%.1f GB activations per step) >> 126 MB L2; no explicit flush" %
                             (P * 1.2 + 4.0),
                       "operands": "fp16 operands (11-bit significand), fp32 accumulation / residual stream / softmax",
                       "ar_steps": ar_steps,
                       "weights": "seeded random init (from_pretrained=False)" if args.weights == "random" else
                                  "trained-like synthetic (synth.peaked_parseq_state_dict)",
                       "crops": "cut on the GPU from the resident pages (ytk_extract_crops_u8, bit-exact with OpenCV)",
                       "recognizer_phase_ms": phase_value},
            "crops_per_s": crops_all * args.steps / (rec_ms / 1e3),
            "det_pages_per_s": world * P * args.steps / (det_ms / 1e3),
            "exchange": {"bytes_sent_per_step_all_ranks": xbytes_all / args.steps,
                         "ms_per_step_max_rank": float(cmax[2].item()) / args.steps,
                         "calls_per_step": x_value["exchange_calls"] / args.steps,
                         "plan_ms_per_step_rank0": x_value.get("plan_ms", 0.0) / args.steps,
                         "results_ms_per_step_rank0": x_value.get("results_ms", 0.0) / args.steps,
                         "path": "device uint8 canvases, ONE torch.distributed all_to_all_single over NCCL per step (no host "
                                 "staging); costs / assignment / descriptors and the returned ids / probabilities travel over "
                                 "host-side gloo groups; ms = host time around the enqueue"},
            "roofline": {"bound": "tensor",
                         "achieved": g_tf / (g_ms / 1e3), "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": g_tf / (g_ms / 1e3) / pk["bf16_tflops_sustained"],
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "gemm_tc_kernel (tcgen05 implicit GEMM): every launch of one step (DBNet convs + "
                                   "PARSeq linears), algorithmic FLOPs (2*M*N*K per launch) over the sum of the launch "
                                   "durations; CUDA events around every launch on the launching stream, one "
                                   "instrumented step right after the timed region",
                         "launches_per_step": g_det["launches"] + g_rec["launches"],
                         "kernel_ms_per_step": g_ms,
                         "share_of_step": g_ms / (total_ms / args.steps),
                         "by_model": {"dbnet": g_det, "parseq": g_rec},
                         "peak_source": pk["source"] + " bf16_tflops_sustained (fp16 and bf16 share the tensor-pipe rate)",
                         "whole_sequence": {"detector": {"achieved": det_tflops,
                                                         "frac": det_tflops / pk["bf16_tflops_sustained"],
                                                         "gflop_per_page": det_flops / P / 1e9},
                                            "recognizer": {"achieved": rec_tflops,
                                                           "frac": rec_tflops / pk["bf16_tflops_sustained"],
                                                           "gflop_per_step_per_gpu": rec_flops_all / world / 1e9},
                                            "step": {"achieved": (det_flops + rec_flops_all / world) * args.steps /
                                                                 (total_ms / 1e3) / 1e12,
                                                     "frac": (det_flops + rec_flops_all / world) * args.steps /
                                                             (total_ms / 1e3) / 1e12 / pk["bf16_tflops_sustained"]}}},
            "cpu_baseline": cpu,
            "e2e": e2e,
            "other_configs": other,
            "gpu_launches": int(launches),
            "clocks": clocks.summary(),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
