#!/usr/bin/env python
"""Cost of the side outputs (adc_match_batch_device_aux), separate from bench.py.

Cone (450x375x64) x 256 pairs and 1242x375x128 x 512 synthetic pairs, device-resident, default engine configuration.
Three arms per shape, alternated round by round in this one process: no side outputs (adc_match_batch_device), all four
(origin, cost_best, cost_second, disp_right), costs only (cost_best, cost_second).  Each batch call is timed with CUDA
events after one warm-up call per arm; maps/s is the median over the rounds.  Also the device time per wave of the plain
WTA kernel and of its side-output instantiation (adc_profile_kernel "wta" / "wta_aux"), and the time one more read of a
wave's volume would take at 7.7 TB/s: the lower bound of a separate min / second-min pass.
The GPU's name and power limit are read in the same run and printed first.  Usage: python tools/confidence_bench.py
"""
import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import adcensus_b200 as A  # noqa: E402
import adc_testlib as T  # noqa: E402

ARMS = {"none": (), "all": ("origin", "cost_best", "cost_second", "disp_right"), "costs": ("cost_best", "cost_second")}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def run(name, pairs, w, h, D, n, rounds):
    idx = [i % len(pairs) for i in range(n)]
    dl = torch.from_numpy(np.stack([pairs[i][0] for i in idx])).cuda()
    dr = torch.from_numpy(np.stack([pairs[i][1] for i in idx])).cuda()
    out = {"disp": torch.empty((n, h, w), dtype=torch.float32, device="cuda"),
           "origin": torch.empty((n, h, w), dtype=torch.uint8, device="cuda"),
           "cost_best": torch.empty((n, h, w), dtype=torch.float32, device="cuda"),
           "cost_second": torch.empty((n, h, w), dtype=torch.float32, device="cuda"),
           "disp_right": torch.empty((n, h, w), dtype=torch.float32, device="cuda")}
    eng = A.Engine(w, h, A.ADCensusOption(max_disparity=D))
    st = torch.cuda.current_stream()

    def call(arm):
        if arm == "none":
            eng.match_batch_device(n, dl.data_ptr(), dr.data_ptr(), out["disp"].data_ptr(), st.cuda_stream)
        else:
            eng.match_batch_device_aux(n, dl.data_ptr(), dr.data_ptr(), out["disp"].data_ptr(), stream=st.cuda_stream,
                                       **{k: out[k].data_ptr() for k in ARMS[arm]})

    ms = {a: [] for a in ARMS}
    for a in ARMS:
        call(a)
    torch.cuda.synchronize()
    ref = out["disp"].clone()
    for _ in range(rounds):
        for a in ARMS:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            call(a)
            e1.record(st)
            torch.cuda.synchronize()
            ms[a].append(e0.elapsed_time(e1))
            assert torch.equal(out["disp"].view(torch.int32), ref.view(torch.int32)), f"{a}: map differs from the plain call's"
    line = {"shape": name, "pairs": n, "wave_pairs": eng.wave_pairs, "lanes": eng.lanes, "rounds": rounds}
    for a in ARMS:
        med = statistics.median(ms[a])
        line[f"{a}_batch_ms"] = round(med, 2)
        line[f"{a}_maps_per_s"] = round(n / med * 1000, 1)
        line[f"{a}_spread_ms"] = [round(min(ms[a]), 2), round(max(ms[a]), 2)]
    for a in ("all", "costs"):
        line[f"{a}_overhead_pct"] = round((line[f"{a}_batch_ms"] / line["none_batch_ms"] - 1) * 100, 2)
    wta, _ = eng.profile_kernel("wta", 20)
    wta_aux, _ = eng.profile_kernel("wta_aux", 20)
    wta2, _ = eng.profile_kernel("wta", 20)
    line["wta_ms_per_wave"] = round(min(wta, wta2), 4)
    line["wta_aux_ms_per_wave"] = round(wta_aux, 4)
    line["volume_read_lower_bound_ms_per_wave"] = round(eng.wave_pairs * w * h * D * 4 / 7.7e12 * 1e3, 4)
    eng.close()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    print(json.dumps(gpu_info()), flush=True)
    run("cone_450x375x64", [T.load_cone()], 450, 375, 64, 256, args.rounds)
    run("1242x375x128", [T.synthetic_pair(1242, 375, 128, 1 + i) for i in range(8)], 1242, 375, 128, 512, args.rounds)


if __name__ == "__main__":
    main()
