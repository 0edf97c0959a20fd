#!/usr/bin/env python
"""Generates tests/golden/golden_wide_cases.json from the UNMODIFIED reference (oracle/_ref): the pins of the disparity
ranges above 256 that an engine reaches with adc_config.max_disparity_range (up to 512).

  cases   sha256 of every tap after every stage for each synthetic pair of WIDE_CASES (the right map's columns the
          reference leaves undefined when min_disparity > 0 are cut off as in make_golden.comparable_tap)
  big     sha256 of the final map of BIG (1242x375, D = 512, seed 1): about a minute of reference time

Run where /root/reference and oracle/_ref exist; the JSON is committed so that machines without them can compare the
oracle and the CUDA path with the real reference's outputs.
"""
import json
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
import adc_testlib as T  # noqa: E402
import make_golden as G  # noqa: E402

# (W, H, option overrides incl. the disparity interval, seed)
WIDE_CASES = [
    (260, 30, {"max_disparity": 257}, 41),                                    # K = 9, padded stride
    (320, 40, {"max_disparity": 400}, 42),                                    # K = 13, padded
    (300, 32, {"max_disparity": 512}, 43),                                    # K = 16, D == 32 * K; D > W
    (256, 48, {"min_disparity": -64, "max_disparity": 320}, 44),              # D = 384, negative dmin
    (200, 60, {"min_disparity": 10, "max_disparity": 300}, 45),               # dmin > 0
    (200, 60, {"max_disparity": 288, "cross_L1": 20, "cross_L2": 9, "so_tso": 25, "irv_ts": 10,
               "do_discontinuity_adjustment": 1}, 46),                        # non-default options, discontinuity adjustment
    (200, 60, {"max_disparity": 300, "do_lr_check": 0}, 47),
    (200, 60, {"max_disparity": 300, "do_filling": 0}, 48),
    (1000, 20, {"max_disparity": 320}, 49),                                   # cost and aggregation rows cut into segments
]
BIG = (1242, 375, 512, 1)   # W, H, D, seed
JSON = T.GOLDEN_DIR / "golden_wide_cases.json"


def case_key(case):
    w, h, over, seed = case
    return f"{w}x{h}-[{over.get('min_disparity', 0)},{over['max_disparity']})-seed{seed}"


def case_inputs(case):
    w, h, over, seed = case
    opt = T.default_option(**over)
    left, right = T.synthetic_pair(w, h, opt.max_disparity - opt.min_disparity, seed)
    return left, right, opt


def big_inputs():
    w, h, D, seed = BIG
    left, right = T.synthetic_pair(w, h, D, seed)
    return left, right, T.default_option(max_disparity=D)


def main():
    T.build_oracle()
    assert T.have_ref(), "oracle/_ref is required"
    out = {"cases": {}, "big": {}}
    for case in WIDE_CASES:
        left, right, opt = case_inputs(case)
        h, w, _ = left.shape
        t0 = time.time()
        ref = T.Reference(w, h, opt)
        ref.begin(left, right)
        hashes = {}
        for st in T.STAGES:
            ref.step()
            for tap in T.STAGE_TAPS[st]:
                hashes[f"{st}/{tap}"] = T.sha(G.comparable_tap(tap, ref.tap(tap), opt))
        ref.close()
        out["cases"][case_key(case)] = {"input_sha": [T.sha(left), T.sha(right)], "hashes": hashes}
        print(case_key(case), "final", hashes["MEDIAN/DISP_L"][:16], f"{time.time() - t0:.1f}s", flush=True)
    left, right, opt = big_inputs()
    h, w, _ = left.shape
    t0 = time.time()
    ref = T.Reference(w, h, opt)
    final = ref.match(left, right)
    ref.close()
    out["big"] = {"width": w, "height": h, "max_disparity": opt.max_disparity, "seed": BIG[3],
                  "input_sha": [T.sha(left), T.sha(right)], "final_sha": T.sha(final)}
    print("big", w, h, opt.max_disparity, "final", out["big"]["final_sha"][:16], f"{time.time() - t0:.1f}s", flush=True)
    JSON.write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
