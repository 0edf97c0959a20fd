#!/usr/bin/env python
"""Generates tests/golden/golden_*.npz from the UNMODIFIED reference (oracle/_ref built from
/root/reference by oracle/Makefile).  Run in the build container; the fixtures are committed so the
GPU box (no /root/reference) can check against the real reference's outputs.

For every case: sha256 of every tap after every stage (bit-exact pin for all intermediates,
including the cost volumes) plus the full arrays of the small per-pixel maps and the final map.
The synthetic pairs of SYNTH_CASES get the hashes only, in tests/golden/golden_synth_cases.json.
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
import adc_testlib as T  # noqa: E402

CASES = {
    # name: (source, W, H, option overrides, seed or crop)
    "cone_full": ("cone", None, None, {}, None),
    "cone_crop": ("cone", 140, 100, {"max_disparity": 32}, (150, 120)),
    "synth_a": ("synth", 97, 61, {"max_disparity": 24}, 2),
    "synth_b": ("synth", 130, 70, {"max_disparity": 37}, 3),
    "synth_opts": ("synth", 120, 90, {"max_disparity": 48, "lambda_ad": 7, "lambda_census": 20, "so_p1": 0.7,
                                       "so_p2": 2.5, "irv_ts": 10, "irv_th": 0.3, "lrcheck_thres": 0.5,
                                       "cross_L1": 20, "cross_L2": 9}, 11),
    "synth_disc": ("synth", 80, 60, {"max_disparity": 32, "do_discontinuity_adjustment": 1}, 10),
}
FULL_TAPS = {"ARMS", "SUPCNT_H", "SUPCNT_V", "DISP_L", "DISP_R", "MISMATCHES", "OCCLUSIONS", "CENSUS_L"}
# synthetic pairs (W, H, D, option overrides, seed): sha256 of every tap after every stage -> golden_synth_cases.json
SYNTH_CASES = [(70, 50, 20, {}, 21), (64, 40, 16, {"min_disparity": 0, "do_lr_check": 0}, 22),
               (90, 64, 40, {"do_filling": 0}, 23), (33, 30, 48, {}, 24), (9, 9, 8, {}, 25),
               (80, 60, 32, {"min_disparity": 2, "max_disparity": 34}, 31),
               (80, 60, 32, {"min_disparity": -4, "max_disparity": 28}, 32)]


def synth_case_key(case):
    w, h, D, over, seed = case
    return f"{w}x{h}x{D}-seed{seed}"


def synth_case_inputs(case):
    w, h, D, over, seed = case
    opt = T.default_option(**{"max_disparity": D, **over})
    left, right = T.synthetic_pair(w, h, D, seed)
    return left, right, opt


def comparable_tap(tap, a, opt):
    """The part of a tap that the reference defines.  With min_disparity > 0, right pixels x >= W - dmin have no
    candidate column at all: the reference then runs its parabola on an uninitialised cost_local[]
    (ADCensusStereo.cpp:271-300, SURVEY 8a A10) -- whatever the heap held; the restatement writes the integer 0 there.
    Undefined in the reference, so not compared."""
    if tap == "DISP_R" and opt.min_disparity > 0:
        return np.ascontiguousarray(a[:, :a.shape[1] - opt.min_disparity])
    return a


def write_synth_cases():
    out = {}
    for case in SYNTH_CASES:
        left, right, opt = synth_case_inputs(case)
        h, w, _ = left.shape
        ref = T.Reference(w, h, opt)
        ref.begin(left, right)
        hashes = {}
        for st in T.STAGES:
            ref.step()
            for tap in T.STAGE_TAPS[st]:
                hashes[f"{st}/{tap}"] = T.sha(comparable_tap(tap, ref.tap(tap), opt))
        ref.close()
        out[synth_case_key(case)] = {"input_sha": [T.sha(left), T.sha(right)], "hashes": hashes}
        print(synth_case_key(case), "final sha", hashes["MEDIAN/DISP_L"][:16])
    (T.GOLDEN_DIR / "golden_synth_cases.json").write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")


def case_inputs(name):
    src, w, h, over, extra = CASES[name]
    opt = T.default_option(**over)
    if src == "cone":
        left, right = T.load_cone()
        if w is not None:
            left, right = T.crop_pair(left, right, extra[0], extra[1], w, h)
    else:
        left, right = T.synthetic_pair(w, h, opt.max_disparity - opt.min_disparity, extra)
    return left, right, opt


def main():
    assert T.have_ref() or (T.build_oracle() or T.have_ref()), "oracle/_ref is required (build container only)"
    out_dir = T.GOLDEN_DIR
    for name in CASES:
        left, right, opt = case_inputs(name)
        h, w, _ = left.shape
        ref = T.Reference(w, h, opt)
        ref.begin(left, right)
        arrays, hashes = {}, {}
        for st in T.STAGES:
            ref.step()
            for tap in T.STAGE_TAPS[st]:
                a = ref.tap(tap)
                hashes[f"{st}/{tap}"] = T.sha(a)
                if tap in FULL_TAPS and (name != "cone_full" or (st in ("WTA", "MEDIAN") and tap in ("DISP_L", "DISP_R"))):
                    arrays[f"{st}__{tap}"] = a.copy()
        stock = ref.stock_match(left, right)
        assert T.sha(stock) == hashes["MEDIAN/DISP_L"], "staged runner and stock Match disagree"
        np.savez_compressed(out_dir / f"golden_{name}.npz", hashes=json.dumps(hashes), **arrays)
        print(name, w, h, "final sha", hashes["MEDIAN/DISP_L"][:16], "arrays", len(arrays))
    write_synth_cases()


if __name__ == "__main__":
    main()
