#!/usr/bin/env python
"""bench.py -- the contract benchmark of the B200 AD-Census engine.

Metric (BASELINE.json): disparity-maps/sec on Cone 450x375x64, batch 256 per GPU (configs[1]).
A "step" = one pass of the whole hot path (ADCensusStereo::Match for every pair) over one batch of
256 stereo pairs.  Inputs are synthetic in the sense of the contract: the bundled Cone pair
replicated 256x (SURVEY.md 8d, config 2); every output therefore has to equal the oracle's map.

  value : whole-job maps/s with the inputs already resident in HBM (adc_match_batch_device)
  e2e   : the same through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the
          timed region, adc_match_batch_pinned_async + synchronise)
  roofline     : the dominant kernel timed in isolation (CUDA events on the engine's stream)
  cpu_baseline : the reference's own CPU implementation (oracle/_ref) on this box's host cores

`--impl reference` times the reference CPU path (oracle/_ref when it was built, else the oracle
port) with one independent instance per host core, on the same workload/metric.

Multi-GPU: independent pairs shard over the ranks (weak scaling, 256 pairs per rank per step);
NCCL carries only the job descriptor broadcast, the timing max and a result checksum.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

WORKLOAD = "cone_450x375_d64_batch256"
PAIRS_PER_STEP = 256
METRIC = "disparity-maps/sec (450x375x64)"
DUMP_BYTES = 60_000_000     # --dump-outputs stays below 64 MB


def dump_outputs(out_dir: str, disp: np.ndarray) -> None:
    """Writes the [n][H][W] float32 maps of the last timed step to out_dir/disparity.npy: all of them when they fit in
    DUMP_BYTES, else the pairs numpy.random.default_rng(0) picks (sorted), the same ones on every run of a workload."""
    n = disp.shape[0]
    k = max(1, min(n, DUMP_BYTES // disp[0].nbytes))
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    np.save(Path(out_dir) / "disparity.npy", np.ascontiguousarray(disp[idx], dtype=np.float32))


# ------------------------------------------------------------------------------------------------
# reference / CPU arm
def _cpu_worker(args):
    kind, iters = args
    import adc_testlib as T
    left, right = T.load_cone()
    h, w, _ = left.shape
    eng = T.Reference(w, h) if kind == "reference" else T.Oracle(w, h)
    t0 = time.perf_counter()
    eng.time_match(left, right, iters)
    return time.perf_counter() - t0


def cpu_baseline(iters_per_core: int, cores: int | None = None) -> dict:
    """The reference has no threads: the most a box can do with it is one independent single-threaded
    instance per core.  On a many-core host that many instances fight over memory bandwidth, so the
    instance count is scanned (all cores, half, a quarter) and the best aggregate is reported."""
    if cores is None:
        n = os.cpu_count() or 1
        best = None
        tried = {}
        for c in sorted({n, max(1, n // 2), max(1, n // 4)}, reverse=True):
            r = _cpu_baseline_n(iters_per_core, c)
            tried[str(c)] = r["value"]
            if best is None or r["value"] > best["value"]:
                best = r
        best["instances_tried_maps_per_s"] = tried
        return best
    return _cpu_baseline_n(iters_per_core, cores)


def _cpu_baseline_n(iters_per_core: int, cores: int) -> dict:
    import adc_testlib as T
    T.build_oracle()
    kind = "reference" if T.have_ref() else "port"
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        per = pool.map(_cpu_worker, [(kind, iters_per_core)] * cores)
    wall = time.perf_counter() - t0
    busy = max(per)
    return {"value": round(cores * iters_per_core / busy, 4), "unit": "maps/s", "cores": cores, "kind": kind,
            "sample": f"{iters_per_core} Cone 450x375x64 Match calls on each of {cores} independent "
                      f"single-threaded instances ({'oracle/_ref, unmodified reference sources' if kind == 'reference' else 'oracle/adc_oracle.c port'}); "
                      f"slowest instance {busy:.2f}s, wall incl. process start {wall:.2f}s",
            "single_core_s_per_map": round(statistics.median(per) / iters_per_core, 4)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # bounded sample: every "step" = iters_per_core matches on each core.  The instance count (all host threads, half, a
    # quarter -- the single-threaded reference is memory-bound when every hardware thread runs one) is scanned once,
    # untimed; the timed steps then run at the best count, so that the whole arm stays within a few minutes.
    per_step = 1
    scan = cpu_baseline(per_step)
    cores = scan["cores"]
    for _ in range(max(0, args.warmup - 1) and 1 or 0):
        cpu_baseline(per_step, cores)
    t0 = time.perf_counter()
    res = None
    vals = []
    for _ in range(args.steps):
        res = cpu_baseline(per_step, cores)
        vals.append(res["value"])
    res["instances_tried_maps_per_s"] = scan.get("instances_tried_maps_per_s")
    wall = time.perf_counter() - t0
    value = statistics.median(vals)
    res["value"] = value
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "maps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1000 * wall / max(1, args.steps), 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(_config_dict(WORKLOAD, PAIRS_PER_STEP, 450, 375, 64),
                           note="each CPU step is a bounded sample of the workload (one Cone pair per host core)"),
            "cpu_baseline": res,
            "e2e": {"value": value, "unit": "maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_ev = index, [], threading.Event()

    def run(self):
        while not self._stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop_ev.wait(0.2)

    def stop(self) -> dict:
        self._stop_ev.set()
        self.join(timeout=3)
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _config_dict(wl_name, n, w, h, D, eng=None, world=1, pipelined=True, sharded=False):
    """The `config` object of the JSON line -- built the same way by both arms so that the driver can compare them."""
    c = {"workload": wl_name, "pairs_per_step_per_gpu": n, "width": w, "height": h, "disparities": D}
    if eng is not None:
        c.update({"wave_pairs": eng.wave_pairs, "lanes": eng.lanes, "steps_pipelined": pipelined,
                  "l2_policy": "no flush needed: each step streams the whole batch of images and several GB of cost volumes per wave, far beyond the 126 MB L2",
                  "parallelism": (f"dp{world}, one batch owned by rank 0: NCCL scatter of the inputs, per-rank Match, NCCL gather of the maps"
                                  if sharded else f"dp{world} (independent pairs, no data-path collective)")})
    return c


def _golden_final_sha(workload):
    """sha256 of the final map(s) the UNMODIFIED reference produced for this workload's inputs (tests/golden)."""
    import adc_testlib as T
    if workload == "cone":
        z = np.load(T.GOLDEN_DIR / "golden_cone_full.npz")
        return {0: json.loads(str(z["hashes"]))["MEDIAN/DISP_L"]}
    big = json.loads((T.GOLDEN_DIR / "golden_big.json").read_text())
    if workload == "kitti":
        return {0: big["kitti_s1"]["hashes"]["MEDIAN/DISP_L"], 1: big["kitti_s2"]["hashes"]["MEDIAN/DISP_L"]}
    return {0: big["p1080_s1"]["hashes"]["MEDIAN/DISP_L"]}


def reference_single_instance(left, right, dmax):
    """BASELINE.md section 4 step 2: ONE instance of the reference on one otherwise idle core -- Match wall time (median of
    5) and the split over the stages its own timers print (ADCensusStereo.cpp:88-129), taken with the staged runner."""
    import adc_testlib as T
    T.build_oracle()
    kind = "reference" if T.have_ref() else "port"
    h, w, _ = left.shape
    mk = (lambda: T.Reference(w, h, T.default_option(max_disparity=dmax))) if kind == "reference" else \
         (lambda: T.Oracle(w, h, T.default_option(max_disparity=dmax)))
    eng = mk()
    tot = []
    for _ in range(5):
        t0 = time.perf_counter()
        eng.time_match(left, right, 1)
        tot.append(time.perf_counter() - t0)
    groups = {"cost": ["COST"], "aggregation": ["ARMS", "AGG1", "AGG2", "AGG3", "AGG4"], "scanline": ["SO1", "SO2", "SO3", "SO4"],
              "wta": ["WTA"], "refine": ["OUTLIER", "VOTE", "INTERP", "DISC", "MEDIAN"]}
    split = {k: 0.0 for k in groups}
    eng.begin(left, right)
    for st in T.STAGES:
        t0 = time.perf_counter()
        eng.step()
        dt = time.perf_counter() - t0
        for k, v in groups.items():
            if st in v:
                split[k] += dt
    eng.close()
    return {"kind": kind, "cores": 1, "s_per_map_median_of_5": round(statistics.median(tot), 4),
            "stage_s": {k: round(v, 4) for k, v in split.items()}}


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    import adcensus_b200 as A
    import adc_testlib as T

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # workloads: BASELINE.json configs[1] (the contract's metric) by default; configs[2] / configs[3] on request
    seeds = 1
    if args.workload == "cone":
        left, right = T.load_cone()
        dmax_w, n, wl_name = 64, PAIRS_PER_STEP, WORKLOAD
        lefts = rights = None
    else:
        w0, h0, dmax_w, n = (1242, 375, 128, 512) if args.workload == "kitti" else (1920, 1080, 192, 64)
        wl_name = f"synthetic_{w0}x{h0}_d{dmax_w}_batch{n}"
        seeds = 16 if args.workload == "kitti" else 8        # distinct synthetic pairs, cycled through the batch (SURVEY 8d)
        pairs = [T.synthetic_pair(w0, h0, dmax_w, s + 1) for s in range(seeds)]
        lefts = np.stack([pairs[i % seeds][0] for i in range(n)])
        rights = np.stack([pairs[i % seeds][1] for i in range(n)])
        left, right = pairs[0]
    if args.pairs > 0:
        n = args.pairs
        if lefts is not None:
            lefts = np.stack([pairs[i % seeds][0] for i in range(n)])
            rights = np.stack([pairs[i % seeds][1] for i in range(n)])
    h, w, _ = left.shape
    # job descriptor from rank 0 (the only data-path collective besides the final reductions)
    desc = torch.tensor([w, h, 0, dmax_w, n], dtype=torch.int32, device=dev)
    if world > 1:
        dist.broadcast(desc, src=0)
    w, h, dmin, dmax, n = [int(v) for v in desc.tolist()]

    opt = A.ADCensusOption(min_disparity=dmin, max_disparity=dmax)
    eng = A.Engine(w, h, opt, device=local, wave_pairs=args.wave_pairs, lanes=args.lanes)
    eng.set_pipelined(not args.no_pipeline)
    N = w * h
    np_left = np.repeat(left[None], n, 0) if lefts is None else lefts
    np_right = np.repeat(right[None], n, 0) if rights is None else rights
    h_left = torch.from_numpy(np_left).pin_memory()
    h_right = torch.from_numpy(np_right).pin_memory()
    h_disp = torch.empty((n, h, w), dtype=torch.float32).pin_memory()
    d_left, d_right = h_left.to(dev), h_right.to(dev)
    d_disp = torch.empty((n, h, w), dtype=torch.float32, device=dev)
    st = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, join=True):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count
        e0.record(st)
        for _ in range(steps):
            fn()
        if join:
            eng.join(st.cuda_stream)    # pipelined engine: the K steps flow into each other, the join is inside the timed region
        e1.record(st)
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        launches = torch.tensor([eng.launch_count - l0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.all_reduce(launches, op=dist.ReduceOp.SUM)
        barrier()
        return float(ms.item()), int(launches.item())

    if args.sharded:
        return run_sharded_arm(args, eng, dev, rank, world, n, w, h, dmax - dmin, wl_name, np_left, np_right, timed, barrier)

    dev_step = lambda: eng.match_batch_device(n, d_left.data_ptr(), d_right.data_ptr(), d_disp.data_ptr(), st.cuda_stream)
    e2e_step = lambda: eng.match_batch_pinned_async(n, h_left.data_ptr(), h_right.data_ptr(), h_disp.data_ptr(), st.cuda_stream)

    for _ in range(max(3, args.warmup)):
        dev_step()
    eng.join(st.cuda_stream)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ms_dev, launches = timed(dev_step, args.steps)
    clocks = sampler.stop() if sampler else None
    for _ in range(2):
        e2e_step()
    eng.join(st.cuda_stream)
    ms_e2e, _ = timed(e2e_step, args.steps)

    # correctness guard inside the bench: the maps of the timed runs against the sha256 of the map the UNMODIFIED
    # reference produced for the same input (tests/golden, generated by tools/make_golden*.py from oracle/_ref);
    # every other copy of a pair must equal the checked one, and the device and host paths must agree
    golden = _golden_final_sha(args.workload)
    hd, dd = h_disp.numpy(), d_disp.cpu().numpy()
    ok = all(T.sha(hd[i]) == sha for i, sha in golden.items())
    for s0 in range(min(seeds, n)):
        ok = ok and bool((hd[s0::seeds].view(np.uint32) == hd[s0].view(np.uint32)[None]).all())
    okd = bool(np.array_equal(dd.view(np.uint32), hd.view(np.uint32)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dd)
    flag = torch.tensor([int(ok and okd)], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)

    line = None
    if rank == 0:
        # ---- the reference's contract literally: pageable host buffers through the synchronous batch call
        eng.set_pipelined(False)
        pg_disp = np.empty((n, h, w), np.float32)
        eng._L.adc_match_batch_strided(eng._h, n, np_left.ctypes.data, np_right.ctypes.data, pg_disp.ctypes.data)   # warm-up
        t0 = time.perf_counter()
        reps_pg = max(1, min(args.steps, 3))
        for _ in range(reps_pg):
            rc = eng._L.adc_match_batch_strided(eng._h, n, np_left.ctypes.data, np_right.ctypes.data, pg_disp.ctypes.data)
        t_pg = (time.perf_counter() - t0) / reps_pg
        pageable = {"value": round(n / t_pg, 2), "unit": "maps/s", "ms_per_step": round(1000 * t_pg, 3),
                    "call": "adc_match_batch_strided on pageable numpy arrays (host wall clock; staging through the engine's pinned ring)",
                    "bit_identical": bool(rc == 0 and np.array_equal(pg_disp.view(np.uint32), hd.view(np.uint32)))}
        # ---- one pair at a time: ADCensusStereo::Match as the reference's caller uses it (main.cpp:118)
        lat, stages = [], []
        for _ in range(25):
            t0 = time.perf_counter()
            eng.match(left, right)
            lat.append(1000 * (time.perf_counter() - t0))
            stages.append(eng.last_stage_ms())
        lat, stages = lat[5:], stages[5:]
        single = {"match_ms_median_of_20": round(statistics.median(lat), 3),
                  "stage_ms_median": dict(zip(("cost", "aggregation", "scanline", "wta", "refine", "copy_out"),
                                              [round(statistics.median(c), 3) for c in zip(*stages)])),
                  "note": "adc_match: pageable host pointers in, host map out, synchronous; stage times from CUDA events"}
        eng.set_pipelined(not args.no_pipeline)

        peaks = {}
        pk = ROOT / "MEASURED_PEAKS.json"
        if pk.exists():
            peaks = json.loads(pk.read_text())
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        V, Nf = 4.0 * N * (dmax - dmin), float(N)
        kern = {}
        names = ["cost_volume", "arm_sum_h", "arm_sum2_v", "arm_sum2_h", "arm_sum_h_div", "arm_sum_v_div", "scanline_x", "scanline_y", "wta"]
        for name in names:
            try:
                kms, kbytes = eng.profile_kernel(name, reps=5)
            except A.AdcError:
                continue
            kern[name] = {"ms_per_launch": round(kms, 4), "algorithmic_bytes": kbytes,
                          "achieved_gbs": round(kbytes / (kms * 1e-3) / 1e9, 1),
                          "frac": round(kbytes / (kms * 1e-3) / 1e9 / hbm_peak, 4), "pairs_per_launch": eng.wave_pairs}
        # Aggregation STAGE on SURVEY 8(d)'s bytes: (2V + 6N) per ITERATION (the first-pass result is an on-chip intermediate
        # in that model), four iterations, against the time of ALL its launches of a wave (kernels timed alone, CUDA events).
        fused = "arm_sum2_v" in kern and "arm_sum2_h" in kern
        if fused:
            agg_ms = (kern["arm_sum_h"]["ms_per_launch"] + 2 * kern["arm_sum2_v"]["ms_per_launch"] +
                      kern["arm_sum2_h"]["ms_per_launch"] + kern["arm_sum_h_div"]["ms_per_launch"])
            agg_launches, agg_transfers = 5, 10
        else:
            agg_ms = 4 * (kern["arm_sum_h"]["ms_per_launch"] + kern["arm_sum_v_div"]["ms_per_launch"])
            agg_launches, agg_transfers = 8, 16
        agg_bytes = 4 * (2 * V + 6 * Nf) * eng.wave_pairs
        aggregation = {"model": "SURVEY 8(d): (2V + 6N) per iteration x 4 iterations per pair", "launches_per_wave": agg_launches,
                       "volume_transfers_per_pair": agg_transfers, "ms_per_wave": round(agg_ms, 4),
                       "achieved_gbs": round(agg_bytes / (agg_ms * 1e-3) / 1e9, 1),
                       "frac": round(agg_bytes / (agg_ms * 1e-3) / 1e9 / hbm_peak, 4)}
        so_ms = 2 * (kern["scanline_x"]["ms_per_launch"] + kern["scanline_y"]["ms_per_launch"])
        # dominant kernel of a step = the launch kind with the largest share of device time
        if fused:
            share = {"arm_sum2_v": 2 * kern["arm_sum2_v"]["ms_per_launch"], "arm_sum2_h": kern["arm_sum2_h"]["ms_per_launch"],
                     "scanline_x": so_ms / 2, "scanline_y": so_ms / 2}
        else:
            share = {"arm_sum_v_div": agg_ms / 2, "arm_sum_h": agg_ms / 2, "scanline_x": so_ms / 2, "scanline_y": so_ms / 2}
        dom = max(share, key=share.get)
        # measured DRAM bytes of that kernel (ncu --set full capture summarised in profiles/; per pair there, per launch here)
        traffic, tsrc = None, None
        tf = ROOT / "profiles" / "traffic.json"
        if tf.exists():
            tj = json.loads(tf.read_text())
            per_pair = tj.get(dom, {}).get("dram_bytes_per_pair")
            tsrc = tj.get("_source")
            if per_pair:
                traffic = round(per_pair * eng.wave_pairs)
        roof = {"kernel": dom, "bound": "hbm", "achieved": kern[dom]["achieved_gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": kern[dom]["frac"], "traffic": traffic, "peak_source": peak_src,
                "note": "algorithmic bytes per launch = (2V + 6N) per pair x pairs per launch, V = 4*H*W*D: the kernel reads one volume and "
                        "writes one (a fused double pass keeps its intermediate in shared memory; it does one iteration's worth of work per "
                        "launch, SURVEY 8d); traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture "
                        f"({tsrc}); kernel timed alone with CUDA events on the engine's stream; 'aggregation' below is the whole stage on the 8(d) model"}
        total_maps = world * n * args.steps
        value = total_maps / (ms_dev * 1e-3)
        e2e_v = total_maps / (ms_e2e * 1e-3)
        b_map = 18.0 * 4.0 * N * (dmax - dmin)
        cpu = cpu_baseline(1) if (world == 1 and not args.no_cpu and args.workload == "cone") else None
        metric = METRIC if args.workload == "cone" else f"disparity-maps/sec ({w}x{h}x{dmax - dmin})"
        line = {"metric": metric, "value": round(value, 2), "unit": "maps/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": round(ms_dev / args.steps, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": _config_dict(wl_name, n, w, h, dmax - dmin, eng, world, not args.no_pipeline),
                "e2e": {"value": round(e2e_v, 2), "unit": "maps/s", "h2d_bytes_per_step": n * 2 * N * 3,
                        "d2h_bytes_per_step": n * N * 4, "ms_per_step": round(ms_e2e / args.steps, 3),
                        "call": "adc_match_batch_pinned_async on pinned host buffers + adc_join"},
                "e2e_pageable": pageable, "single_pair": single,
                "gpu_launches": launches, "clocks": clocks, "outputs_bit_identical": bool(flag.item()),
                "outputs_checked_against": "sha256 of the unmodified reference's map (tests/golden), every copy, device and host path",
                "pipeline_hbm": {"algorithmic_bytes_per_map": b_map, "achieved_gbs": round(value * b_map / 1e9 / world, 1),
                                 "frac": round(value * b_map / 1e9 / world / hbm_peak, 4)},
                "roofline": roof, "aggregation": aggregation, "kernels": kern}
        if cpu:
            cpu["single_instance"] = reference_single_instance(left, right, dmax)
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def run_sharded_arm(args, eng, dev, rank, world, n, w, h, D, wl_name, np_left, np_right, timed, barrier):
    """BASELINE.json configs[4]: ONE batch of n x world pairs owned by rank 0 (resident in its HBM), scattered over the
    ranks with NCCL, matched by every rank's engine, the maps gathered back on rank 0 with NCCL (SURVEY 8e).  A step =
    scatter + Match + gather of the whole batch; value = pairs / max-over-ranks time."""
    import torch
    import torch.distributed as dist
    import adc_testlib as T
    from adcensus_b200.parallel import run_sharded_device
    N, total = w * h, n * world
    seeds = 16 if args.workload == "kitti" else (8 if args.workload == "1080p" else 1)
    st = torch.cuda.current_stream()
    d_l = d_r = d_out = None
    if rank == 0:
        reps = (total + n - 1) // n
        d_l = torch.from_numpy(np_left).to(dev).repeat((reps, 1, 1, 1))[:total].contiguous()   # n is a multiple of the seed cycle
        d_r = torch.from_numpy(np_right).to(dev).repeat((reps, 1, 1, 1))[:total].contiguous()
        d_out = torch.empty((total, h, w), dtype=torch.float32, device=dev)
    phases = {}
    step = lambda: run_sharded_device(eng, d_l, d_r, d_out, total, h, w, dev, phases)
    for _ in range(max(1, args.warmup)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches = timed(step, args.steps, join=False)
    clocks = sampler.stop() if sampler else None
    if "resolve" in phases:
        phases["resolve"]()
    ok, check = True, {}
    if rank == 0:
        golden = _golden_final_sha(args.workload)
        out = d_out.cpu().numpy()
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, out)
        check["golden"] = all(T.sha(out[i]) == sha for i, sha in golden.items())
        bad = [int(i) for i in range(total) if not np.array_equal(out[i].view(np.uint32), out[i % seeds].view(np.uint32))]
        check["copies_equal"] = not bad
        if bad:
            check["differing_pairs"] = len(bad)
            check["first_differing"] = bad[:4]
        ok = check["golden"] and check["copies_equal"]
    flag = torch.tensor([int(ok)], dtype=torch.int32, device=dev)
    ph = torch.tensor([phases.get("scatter_ms", 0.0), phases.get("compute_ms", 0.0), phases.get("gather_ms", 0.0)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.all_reduce(ph, op=dist.ReduceOp.MAX)
    if rank == 0:
        value = total * args.steps / (ms * 1e-3)
        metric = METRIC if args.workload == "cone" else f"disparity-maps/sec ({w}x{h}x{D})"
        line = {"metric": metric, "value": round(value, 2), "unit": "maps/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(1, args.warmup), "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": dict(_config_dict(wl_name, n, w, h, D, eng, world, False, sharded=True), batch_owned_by_rank0=total),
                "sharded": {"total_pairs": total, "scatter_bytes": (total - n) * 2 * N * 3, "gather_bytes": (total - n) * N * 4,
                            "last_step_ms_max_over_ranks": {"scatter": round(float(ph[0]), 3), "compute": round(float(ph[1]), 3),
                                                            "gather": round(float(ph[2]), 3)},
                            "note": "inputs and results resident in rank 0's HBM; NCCL point-to-point scatter / gather; phases timed with CUDA events "
                                    "on each rank's stream (the phases of different ranks overlap, so they do not add up to the step)"},
                "gpu_launches": launches, "clocks": clocks, "outputs_bit_identical": bool(flag.item()), "outputs_check": check,
                "outputs_checked_against": "sha256 of the unmodified reference's maps (tests/golden) + every copy of a pair equal, gathered order"}
        print(json.dumps(line), flush=True)
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--wave-pairs", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="join the stream after every step (adc_set_pipelined off): each step then drains the engine")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per step per GPU (default: the BASELINE batch of the workload)")
    ap.add_argument("--sharded", action="store_true",
                    help="BASELINE configs[4] form: one batch of pairs x gpus owned by rank 0, NCCL scatter -> Match -> NCCL gather")
    ap.add_argument("--workload", default="cone", choices=["cone", "kitti", "1080p"],
                    help="cone = BASELINE configs[1] (the contract metric); kitti / 1080p = configs[2] / configs[3] (extra lines)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the disparity maps of the last timed (device-resident) step to "
                         "DIR/disparity.npy, float32 [k][H][W]: the whole batch, or a fixed sample of it below 64 MB")
    args = ap.parse_args()
    if args.dump_outputs:
        if args.impl == "reference":
            ap.error("--dump-outputs writes the GPU path's maps; the reference arm keeps none")
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_gpu_arm(args)


if __name__ == "__main__":
    sys.exit(main())
