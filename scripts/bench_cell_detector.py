"""Throughput of the cell detector's model (RT-DETRv2 at 960 x 960 with 1500 queries, reference
configs/cfg_table_cell_parser_rtdtrv2.py) on one GPU, and the time of its query selection kernel.  Prints one JSON line:

  gpu / power_limit_w        the card and its power limit, read in the same call as the timings
  images_per_s / ms_per_call forward at batch 1 and 8: inputs and outputs resident in HBM, CUDA events around `steps`
                             calls after `warmup` calls, random weights (the timing does not depend on them)
  gflop_per_image            ytk_rtdetr_flops (the GEMMs and attention products of the launch plan)
  device_bytes               activation buffers of the batch-1 / batch-8 launch plans
  topk_us                    ytk_op_rt_topk_f32 at 18900 scores / k = 1500 per image (batch 1 and 8), CUDA events
                             around `topk_launches` back-to-back launches
Usage: python scripts/bench_cell_detector.py [--steps 20] [--warmup 5]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    name, limit = (r.stdout.strip().split(", ") + ["?", "?"])[:2]
    return name, limit


def event_ms(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--topk-launches", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cell_detector.py needs a GPU")
    from yomitoku_b200 import _lib
    from yomitoku_b200.config import TableCellParserRTDETRv2Config, to_config
    from yomitoku_b200.models import RTDETRv2
    L = _lib.lib()
    m = RTDETRv2(cfg=to_config(TableCellParserRTDETRv2Config())).to("cuda")
    S, Q, C = m.img_size, m.num_queries, m.num_classes
    out = {"metric": "images/sec (cell detector RT-DETRv2 forward, %dx%d, %d queries)" % (S, S, Q)}
    name, limit = gpu_info()
    out["gpu"], out["power_limit_w"] = name, limit
    fwd = {}
    for batch in (1, 8):
        x = torch.rand(batch, 3, S, S, device="cuda")
        lg = torch.empty((batch, Q, C), dtype=torch.float32, device="cuda")
        bx = torch.empty((batch, Q, 4), dtype=torch.float32, device="cuda")

        def step():
            _lib.check(L.ytk_rtdetr_forward_f32(m._ensure(), x.data_ptr(), 1, batch, lg.data_ptr(), bx.data_ptr(), 1,
                                                None))
        ms = event_ms(step, args.steps, args.warmup)
        fwd[batch] = {"images_per_s": batch / (ms / 1e3), "ms_per_call": ms,
                      "gflop_per_image": m.flops(batch) / batch / 1e9, "device_bytes": m.device_bytes(batch)}
    out["forward"] = fwd
    out["value"], out["unit"] = fwd[8]["images_per_s"], "images/s (batch 8)"
    topk = {}
    for n in (1, 8):
        scores = torch.randn(n, 18900, device="cuda")
        idx = torch.empty((n, 1500), dtype=torch.int32, device="cuda")

        def sel():
            _lib.check(L.ytk_op_rt_topk_f32(ctypes.c_void_p(scores.data_ptr()), n, 18900, 1500,
                                            ctypes.c_void_p(idx.data_ptr()), None))
        topk["batch%d" % n] = event_ms(sel, args.topk_launches, 10) * 1e3
    out["topk_us"] = topk
    out["steps"], out["warmup"] = args.steps, args.warmup
    print(json.dumps(out))


if __name__ == "__main__":
    main()
