"""CPU tests of the oracle (test infrastructure): pinned against the real reference (oracle/_ref,
where it exists) and against the committed golden vectors produced by the real reference."""
import json
import sys
from pathlib import Path

import numpy as np
import pytest

import adc_testlib as T

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import make_golden as G  # noqa: E402  (case definitions shared with the fixture generator)

FAST_CASES = ["cone_crop", "synth_a", "synth_b", "synth_opts", "synth_disc"]


def _golden(name):
    z = np.load(T.GOLDEN_DIR / f"golden_{name}.npz")
    return json.loads(str(z["hashes"])), z


@pytest.mark.parametrize("name", FAST_CASES)
def test_oracle_matches_golden(name):
    """Every tap after every stage: sha256 equal to what the unmodified reference produced."""
    left, right, opt = G.case_inputs(name)
    hashes, z = _golden(name)
    h, w, _ = left.shape
    orc = T.Oracle(w, h, opt)
    orc.begin(left, right)
    for st in T.STAGES:
        orc.step()
        for tap in T.STAGE_TAPS[st]:
            a = orc.tap(tap)
            assert T.sha(a) == hashes[f"{st}/{tap}"], f"{name}: {st}/{tap} differs from the reference's golden hash"
            key = f"{st}__{tap}"
            if key in z.files:
                assert np.array_equal(a.view(np.uint8), z[key].view(np.uint8)), f"{name}: {key} array differs"


def test_oracle_cone_final_matches_golden(cone):
    """Full-size Cone (BASELINE config 1): final map bit-identical to the reference's
    (sha256 77d70a58d1aa5c71..., also recorded in SURVEY.md 8c)."""
    left, right = cone
    hashes, z = _golden("cone_full")
    h, w, _ = left.shape
    orc = T.Oracle(w, h)
    disp = orc.match(left, right)
    assert T.sha(disp) == hashes["MEDIAN/DISP_L"]
    assert hashes["MEDIAN/DISP_L"].startswith("77d70a58d1aa5c71")
    assert np.array_equal(disp.view(np.uint32), z["MEDIAN__DISP_L"].view(np.uint32))


@pytest.mark.parametrize("case", G.SYNTH_CASES)
def test_oracle_vs_live_reference(case):
    """Every tap after every stage on synthetic pairs (odd sizes, dmin > 0, dmin < 0, options off): sha256 equal to what a
    live run of the unmodified reference produced (golden_synth_cases.json, written by tools/make_golden.py)."""
    g = json.loads((T.GOLDEN_DIR / "golden_synth_cases.json").read_text())[G.synth_case_key(case)]
    left, right, opt = G.synth_case_inputs(case)
    assert [T.sha(left), T.sha(right)] == g["input_sha"]
    h, w, _ = left.shape
    orc = T.Oracle(w, h, opt)
    orc.begin(left, right)
    for st in T.STAGES:
        orc.step()
        for tap in T.STAGE_TAPS[st]:
            assert T.sha(G.comparable_tap(tap, orc.tap(tap), opt)) == g["hashes"][f"{st}/{tap}"], f"{st}/{tap}"


def test_gray_exhaustive():
    """All 2^24 BGR triples: uint8(r*0.299 + g*0.587 + b*0.114) in double, no contraction
    (cost_computor.cpp:69).  gray(128,128,128) = 127 is the classic trap."""
    import ctypes
    T.build_oracle()
    lib = ctypes.CDLL(str(T.ORACLE_DIR / "_build" / "libadc_oracle.so"))
    lib.orc_gray.restype = ctypes.c_uint8
    lib.orc_gray.argtypes = [ctypes.c_uint8] * 3
    assert lib.orc_gray(128, 128, 128) == 127
    # vectorised double arithmetic (numpy never contracts) over the full domain, spot-checked against the C function
    v = np.arange(256, dtype=np.float64)
    r, g, b = v[:, None, None] * 0.299, v[None, :, None] * 0.587, v[None, None, :] * 0.114
    gray = ((r + g) + b).astype(np.uint8)       # [r][g][b]
    assert gray[128, 128, 128] == 127 and gray[255, 255, 255] == 255 and gray[0, 0, 0] == 0
    rng = np.random.default_rng(0)
    for rr, gg, bb in rng.integers(0, 256, size=(20000, 3)):
        assert lib.orc_gray(int(bb), int(gg), int(rr)) == gray[rr, gg, bb]


def test_hamming_and_cost_domain():
    import ctypes
    T.build_oracle()
    lib = ctypes.CDLL(str(T.ORACLE_DIR / "_build" / "libadc_oracle.so"))
    lib.orc_hamming64.argtypes = [ctypes.c_uint64, ctypes.c_uint64]
    lib.orc_cost_value.restype = ctypes.c_float
    lib.orc_cost_value.argtypes = [ctypes.c_int] * 4
    rng = np.random.default_rng(1)
    for a, b in rng.integers(0, 2**63, size=(2000, 2), dtype=np.uint64):
        assert lib.orc_hamming64(int(a), int(b)) == bin(int(a) ^ int(b)).count("1")
    # the full 766 x 64 domain of the AD-census cost: range and monotonicity (cost_computor.cpp:110-117)
    tab = np.array([[lib.orc_cost_value(s, hh, 10, 30) for hh in range(64)] for s in range(766)], np.float32)
    assert tab[0, 0] == 0.0 and tab.min() >= 0.0 and tab.max() < 2.0
    assert (np.diff(tab, axis=0) >= 0).all() and (np.diff(tab, axis=1) >= 0).all()
    assert 1.873 < float(tab.max()) < 1.878           # SURVEY.md 8a/A4 measured [0, 1.8734] on data; domain max is 1.8775


def test_synthetic_generator_properties():
    left, right = T.synthetic_pair(200, 60, 64, 1)
    assert left.shape == (60, 200, 3) and left.dtype == np.uint8
    l2, r2 = T.synthetic_pair(200, 60, 64, 1)
    assert np.array_equal(left, l2) and np.array_equal(right, r2)          # deterministic
    assert 100 < left.mean() < 155 and left.std() > 15                      # textured, not flat / not white noise
    # right(x) == left(x + d_band) exactly inside the image, per 25-row band
    for y in (0, 30, 55):
        found = any(np.array_equal(left[y, d:], right[y, :200 - d]) for d in range(8, 48))
        assert found
