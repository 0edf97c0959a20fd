#!/usr/bin/env python
"""Throughput of engines with a wide disparity range limit (adc_config.max_disparity_range = 512), separate from bench.py.

  1242x375 at D = 256, 384, 512: device-resident batches (maps/s, CUDA events around whole batch calls), the per-kernel
  device time of one wave (adc_profile_kernel) and the six stage times of a single-pair Match (adc_last_stage_ms)
  1920x1080 at D = 400: one device-resident batch

Inputs are synthetic pairs (tests/adc_testlib.synthetic_pair); every volume is far larger than L2.  Prints one JSON line
per configuration; the GPU's name and power limit are read in the same run and printed first.
Usage: python tools/wide_range_bench.py [--reps 3]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import adcensus_b200 as A  # noqa: E402
import adc_testlib as T  # noqa: E402

KERNELS = ("cost_volume", "arm_sum_h", "arm_sum2_v", "arm_sum2_h", "arm_sum_h_div", "scanline_x", "scanline_y", "wta")
STAGES = ("cost", "aggregation", "scanline", "wta", "refine", "output_copy")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def run(w, h, D, n, distinct, wave_pairs, lanes, reps, per_kernel):
    pairs = [T.synthetic_pair(w, h, D, 1 + i) for i in range(distinct)]
    idx = [i % distinct for i in range(n)]
    dl = torch.from_numpy(np.stack([pairs[i][0] for i in idx])).cuda()
    dr = torch.from_numpy(np.stack([pairs[i][1] for i in idx])).cuda()
    dd = torch.empty((n, h, w), dtype=torch.float32, device="cuda")
    eng = A.Engine(w, h, A.ADCensusOption(max_disparity=D), wave_pairs=wave_pairs, lanes=lanes, max_disparity_range=512)
    st = torch.cuda.current_stream()
    eng.match_batch_device(n, dl.data_ptr(), dr.data_ptr(), dd.data_ptr(), st.cuda_stream)   # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(reps):
        eng.match_batch_device(n, dl.data_ptr(), dr.data_ptr(), dd.data_ptr(), st.cuda_stream)
    e1.record(st)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    line = {"shape": f"{w}x{h}x{D}", "pairs": n, "wave_pairs": eng.wave_pairs, "lanes": eng.lanes, "batch_ms": round(ms, 2),
            "maps_per_s": round(n / ms * 1000, 1)}
    if per_kernel:
        line["kernel_ms_per_wave"] = {}
        for name in KERNELS:
            try:
                kms, _ = eng.profile_kernel(name, 5)
                line["kernel_ms_per_wave"][name] = round(kms, 3)
            except A.AdcError:
                line["kernel_ms_per_wave"][name] = None   # not applicable at this size
        for _ in range(3):
            eng.match(*pairs[0])
        line["single_pair_stage_ms"] = dict(zip(STAGES, (round(x, 3) for x in eng.last_stage_ms())))
    eng.close()
    print(json.dumps(line), flush=True)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    print(json.dumps(gpu_info()), flush=True)
    for D in (256, 384, 512):
        run(1242, 375, D, n=48, distinct=8, wave_pairs=8, lanes=3, reps=args.reps, per_kernel=True)
    run(1920, 1080, 400, n=8, distinct=2, wave_pairs=4, lanes=2, reps=args.reps, per_kernel=False)


if __name__ == "__main__":
    main()
