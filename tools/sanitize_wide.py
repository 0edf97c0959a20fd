"""Small wide-range cases (engine limit 512) for compute-sanitizer: K = 9 padded, K = 13 padded, K = 16 full with D > W,
a negative dmin -- through Match and a batch of two waves, each map against the oracle."""
import sys
from pathlib import Path
import numpy as np
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import adcensus_b200 as A
import adc_testlib as T

cases = [(96, 20, 0, 257, 41), (80, 16, 0, 400, 42), (64, 16, 0, 512, 43), (72, 24, -64, 320, 44)]
for (w, h, dmin, dmax, seed) in cases:
    left, right = T.synthetic_pair(w, h, dmax - dmin, seed)
    eng = A.Engine(w, h, A.ADCensusOption(min_disparity=dmin, max_disparity=dmax), wave_pairs=2, lanes=2,
                   max_disparity_range=512)
    a = eng.match(left, right)
    b = eng.match_batch(np.stack([left] * 3), np.stack([right] * 3))
    assert (b.view(np.uint32) == a.view(np.uint32)[None]).all()
    want = T.Oracle(w, h, T.default_option(min_disparity=dmin, max_disparity=dmax)).match(left, right)
    assert a.tobytes() == want.tobytes(), (w, h, dmin, dmax)
    eng.close()
    print("ok", w, h, dmin, dmax, flush=True)
print("all ok")
