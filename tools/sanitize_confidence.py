"""Small side-output cases for compute-sanitizer: adc_match_aux with all four outputs on the default path (push voting),
with cross_L1 > 127 (byte-state voting), at D = 300 (float-state voting, engine limit 512), without the LR check,
without filling and with dmin < 0; then a host batch of three pairs over two waves on two lanes.  Each map against the
oracle, each side output against the oracle-derived one."""
import sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests")); sys.path.insert(0, str(ROOT / "tools"))
import adcensus_b200 as A
import adc_testlib as T
import make_golden_aux as GA

cases = [(64, 40, {"max_disparity": 24}, 81),
         (48, 64, {"max_disparity": 16, "cross_L1": 130, "cross_L2": 17, "cross_t1": 300, "cross_t2": 300}, 82),
         (96, 20, {"max_disparity": 300}, 83),
         (64, 40, {"max_disparity": 24, "do_lr_check": 0}, 84),
         (64, 40, {"max_disparity": 24, "do_filling": 0}, 85),
         (64, 40, {"min_disparity": -8, "max_disparity": 16}, 86)]
for (w, h, over, seed) in cases:
    opt = T.default_option(**over)
    left, right = T.synthetic_pair(w, h, opt.max_disparity - opt.min_disparity, seed)
    o = A.ADCensusOption(**{k: v for k, v in over.items()})
    eng = A.Engine(w, h, o, wave_pairs=2, lanes=2, max_disparity_range=512 if opt.max_disparity > 256 else 0)
    disp, aux = eng.match_aux(left, right)
    want = GA.derive_aux(T.Oracle(w, h, opt), left, right, opt)
    assert disp.tobytes() == want["disp"].tobytes(), (w, h, over)
    for k in ("origin", "cost_best", "cost_second", "disp_right"):
        assert aux[k].tobytes() == want[k].tobytes(), (w, h, over, k)
    db, ab = eng.match_batch_aux(np.stack([left] * 3), np.stack([right] * 3))
    for k in ("origin", "cost_best", "cost_second", "disp_right"):
        assert (ab[k] == aux[k][None]).all(), (w, h, over, k)
    eng.close()
    print("ok", w, h, over, flush=True)
print("all ok")
