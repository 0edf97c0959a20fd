#!/usr/bin/env python
"""Generates tests/golden/golden_aux.json from the UNMODIFIED reference (oracle/_ref): sha256 of the side outputs
(adc_aux_outputs: origin, cost_best, cost_second, disp_right) of every case in AUX_CASES.

The side outputs are pure functions of the staged runner's taps (derive_aux below, which the tests also apply to the
oracle):
  cost_best    min over d of VOL_AGGR after SO4 (the volume WTA scans)
  cost_second  min over the d with |d - b| >= 2, b = the first minimum; +inf where there is none
  origin       from DISP_L after WTA (the WTA-invalid flag), the MISMATCHES / OCCLUSIONS lists after OUTLIER and after
               VOTE, and DISP_L after INTERP (after OUTLIER without filling)
  disp_right   DISP_R after WTA, with make_golden.comparable_tap's rule for the columns undefined when dmin > 0

Run where the reference harness oracle/_ref has been built; the JSON is committed.
"""
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
import adc_testlib as T  # noqa: E402
import make_golden as G  # noqa: E402

# ADC_ORIGIN_* (include/adcensus_b200.h)
MATCHED, INVALID, WTA_INVALID = 0, 5, 8

# ("golden", name of make_golden.CASES) or ("synth", (W, H, D, option overrides, seed)) as in make_golden.SYNTH_CASES
AUX_CASES = ([("golden", "cone_full"), ("golden", "synth_disc")]            # defaults; discontinuity adjustment on
             + [("synth", c) for c in G.SYNTH_CASES]                        # lr check off, filling off, dmin > 0, dmin < 0
             + [("synth", (60, 120, 16, {"cross_L1": 130, "cross_L2": 17, "cross_t1": 300, "cross_t2": 300}, 61)),
                ("synth", (200, 40, 300, {}, 62)),                          # D = 300: needs the wide limit
                ("synth", (40, 30, 3, {"min_disparity": -1, "max_disparity": 2}, 63)),     # range 3: cost_second is +inf
                ("synth", (40, 30, 3, {"do_lr_check": 0}, 64))])       # where b = 1; WTA-invalid pixels without the LR check
JSON = T.GOLDEN_DIR / "golden_aux.json"


def case_key(case):
    kind, spec = case
    return spec if kind == "golden" else G.synth_case_key(spec)


def case_inputs(case):
    kind, spec = case
    return G.case_inputs(spec) if kind == "golden" else G.synth_case_inputs(spec)


def _label_map(lists, h, w):
    """Outlier class per pixel (0, 1 = mismatch, 2 = occlusion) from the MISMATCHES / OCCLUSIONS taps."""
    lab = np.zeros((h, w), np.uint8)
    for k, xy in enumerate(lists):
        lab[xy[:, 1], xy[:, 0]] = k + 1
    return lab


def costs_from_volume(vol):
    """(cost_best, cost_second) of an [H][W][D] volume."""
    b = vol.argmin(axis=2)                       # first minimum, as WTA's strict '>'
    best = np.take_along_axis(vol, b[:, :, None], axis=2)[:, :, 0]
    far = np.abs(np.arange(vol.shape[2])[None, None, :] - b[:, :, None]) >= 2
    second = np.where(far, vol, np.float32(np.inf)).min(axis=2).astype(np.float32)
    return np.ascontiguousarray(best), np.ascontiguousarray(second)


def derive_aux(checker, left, right, opt):
    """Runs a staged checker (T.Oracle or T.Reference) through the whole pipeline and returns the side outputs and the
    final map, as the library defines them."""
    h, w, _ = left.shape
    checker.begin(left, right)
    taps = {}
    want = {"SO4": ["VOL_AGGR"], "WTA": ["DISP_L", "DISP_R"], "OUTLIER": ["DISP_L", "MISMATCHES", "OCCLUSIONS"],
            "VOTE": ["MISMATCHES", "OCCLUSIONS"], "INTERP": ["DISP_L"], "MEDIAN": ["DISP_L"]}
    for st in T.STAGES:
        checker.step()
        for tap in want.get(st, []):
            taps[f"{st}/{tap}"] = checker.tap(tap).copy()
    best, second = costs_from_volume(taps["SO4/VOL_AGGR"])
    lab0 = _label_map([taps["OUTLIER/MISMATCHES"], taps["OUTLIER/OCCLUSIONS"]], h, w)
    lab1 = _label_map([taps["VOTE/MISMATCHES"], taps["VOTE/OCCLUSIONS"]], h, w)
    final = taps["INTERP/DISP_L"] if opt.do_filling else taps["OUTLIER/DISP_L"]
    origin = np.where(lab1 == 0, lab0, lab0 + 2).astype(np.uint8)
    origin = np.where(np.isinf(final), np.uint8(INVALID), origin).astype(np.uint8)
    origin |= np.where(np.isinf(taps["WTA/DISP_L"]), np.uint8(WTA_INVALID), np.uint8(0))
    return {"origin": origin, "cost_best": best, "cost_second": second, "disp_right": taps["WTA/DISP_R"],
            "disp": taps["MEDIAN/DISP_L"]}


def aux_hashes(aux, opt):
    out = {k: T.sha(aux[k]) for k in ("origin", "cost_best", "cost_second", "disp")}
    out["disp_right"] = T.sha(G.comparable_tap("DISP_R", aux["disp_right"], opt))
    return out


def main():
    T.build_oracle()
    assert T.have_ref(), "oracle/_ref is required"
    out = {}
    for case in AUX_CASES:
        left, right, opt = case_inputs(case)
        h, w, _ = left.shape
        ref = T.Reference(w, h, opt)
        aux = derive_aux(ref, left, right, opt)
        ref.close()
        out[case_key(case)] = {"input_sha": [T.sha(left), T.sha(right)], "hashes": aux_hashes(aux, opt),
                               "origin_counts": {int(k): int(v) for k, v in zip(*np.unique(aux["origin"], return_counts=True))}}
        print(case_key(case), out[case_key(case)]["origin_counts"], flush=True)
    JSON.write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")


if __name__ == "__main__":
    main()
