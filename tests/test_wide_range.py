"""Disparity ranges above 256 behind the per-engine limit adc_config.max_disparity_range (up to 512).

CPU: the adc_config layout and its Python mirror, the limit's argument checks (they fail before any device work), and
the oracle against the unmodified reference's hashes of every tap after every stage (tests/golden/golden_wide_cases.json,
written by tools/make_golden_wide.py).
GPU: every stage of every wide case against the oracle, a loaded 12-pair wave whose pair offsets pass 2^31 floats, the
limits, and the C++ overload Initialize(width, height, option, max_disparity_range).
"""
import ctypes
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import adc_testlib as T

sys.path.insert(0, str(Path(__file__).resolve().parent.parent / "tools"))
import make_golden as G  # noqa: E402
import make_golden_wide as GW  # noqa: E402

WIDE = 512
CASE_IDS = [GW.case_key(c) for c in GW.WIDE_CASES]


def _golden():
    return json.loads(GW.JSON.read_text())


def _lib():
    import adcensus_b200 as A
    from adcensus_b200.build import build_library
    build_library()
    return A, A.load_library()


def _engine(w, h, opt, **kw):
    import adcensus_b200 as A
    o = A.ADCensusOption()
    for name, _ in T.Option._fields_:
        if not name.startswith("_"):
            setattr(o, name, getattr(opt, name))
    return A.Engine(w, h, o, **kw)


def _same(name, got, want):
    assert got.shape == want.shape, f"{name}: shape {got.shape} vs {want.shape}"
    if got.dtype.kind == "f":
        eq = got.view(np.uint32) == want.view(np.uint32)
        if not eq.all():
            fin = np.isfinite(got) & np.isfinite(want)
            md = float(np.abs(got[fin].astype(np.float64) - want[fin]).max()) if fin.any() else 0.0
            raise AssertionError(f"{name}: {int((~eq).sum())} of {eq.size} values differ, max abs diff {md:.3e}")
    else:
        assert np.array_equal(got, want), f"{name}: {int((got != want).sum())} of {got.size} values differ"


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def test_config_layout_and_mirror():
    A, L = _lib()
    from adcensus_b200.engine import _Config
    assert ctypes.sizeof(_Config) == 64
    offs = {n: getattr(_Config, n).offset for n, _ in _Config._fields_}
    assert offs == {"device": 0, "wave_pairs": 4, "lanes": 8, "debug_flags": 12, "max_disparity_range": 16, "reserved": 20}
    assert _Config.reserved.size == 11 * 4
    hdr = (T.REPO / "include" / "adcensus_b200.h").read_text()
    assert "#define ADC_MAX_DISPARITY_RANGE 256" in hdr and "#define ADC_MAX_DISPARITY_RANGE_WIDE 512" in hdr
    assert (A.engine.MAX_DISPARITY_RANGE, A.engine.MAX_DISPARITY_RANGE_WIDE) == (256, 512)


def _create(L, A, w, h, opt, limit):
    from adcensus_b200.engine import _Config
    cfg = _Config(max_disparity_range=limit)
    hd = ctypes.c_void_p()
    rc = L.adc_create(w, h, ctypes.byref(opt), ctypes.byref(cfg), ctypes.byref(hd))
    if hd.value:
        L.adc_destroy(hd)
    return rc, L.adc_last_error().decode()


def test_limit_rejections_need_no_gpu():
    """The limit is checked before any device work: a bad limit is an argument error, a range above the engine's limit
    is unsupported (and says "disparity range"), whether or not a GPU is present."""
    A, L = _lib()
    o = A.ADCensusOption(max_disparity=64)
    for bad in (-1, WIDE + 1):
        rc, msg = _create(L, A, 64, 48, o, bad)
        assert rc == 1 and "max_disparity_range" in msg, (bad, rc, msg)
    rc, msg = _create(L, A, 64, 48, A.ADCensusOption(max_disparity=WIDE + 1), WIDE)
    assert rc == 3 and "disparity range" in msg, (rc, msg)
    rc, msg = _create(L, A, 64, 48, A.ADCensusOption(min_disparity=-1, max_disparity=300), 300)
    assert rc == 3 and "disparity range 301 > 300" in msg, (rc, msg)
    rc, msg = _create(L, A, 64, 48, A.ADCensusOption(max_disparity=257), 0)      # zero = the default limit of 256
    assert rc == 3 and "disparity range" in msg, (rc, msg)
    s = A.ADCensusStereo()
    assert s.Initialize(64, 48, A.ADCensusOption(max_disparity=300), max_disparity_range=-1) is False
    assert "max_disparity_range" in s.last_error


@pytest.mark.parametrize("case", GW.WIDE_CASES, ids=CASE_IDS)
def test_oracle_vs_reference_wide(case):
    """Every tap after every stage of the oracle hashes to what the unmodified reference produced."""
    g = _golden()["cases"][GW.case_key(case)]
    left, right, opt = GW.case_inputs(case)
    assert [T.sha(left), T.sha(right)] == g["input_sha"]
    h, w, _ = left.shape
    orc = T.Oracle(w, h, opt)
    orc.begin(left, right)
    for st in T.STAGES:
        orc.step()
        for tap in T.STAGE_TAPS[st]:
            assert T.sha(G.comparable_tap(tap, orc.tap(tap), opt)) == g["hashes"][f"{st}/{tap}"], f"{st}/{tap}"


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", GW.WIDE_CASES, ids=CASE_IDS)
def test_stage_parity_wide(case):
    """All sixteen stages, every tap, against the oracle; then match() against the staged result and the reference hash."""
    left, right, opt = GW.case_inputs(case)
    h, w, _ = left.shape
    orc = T.Oracle(w, h, opt)
    eng = _engine(w, h, opt, max_disparity_range=WIDE)
    assert eng.max_disparity_range == WIDE
    orc.begin(left, right)
    for st in T.STAGES:
        orc.step()
        eng.debug_run(left, right, st)
        for tap in T.STAGE_TAPS[st]:
            _same(f"{st}/{tap}", eng.tap(tap), orc.tap(tap))
    out = eng.match(left, right)
    _same("match", out, orc.tap("DISP_L"))
    assert T.sha(out) == _golden()["cases"][GW.case_key(case)]["hashes"]["MEDIAN/DISP_L"]
    eng.close()


@pytest.mark.gpu
def test_large_wave_wide():
    """1242x375 at D = 512, twelve pairs in one wave: the pair offsets of the volumes pass 2^31 floats and the bulk
    scanline ring runs with every SM loaded.  Every map equals its single-pair map; seed 1 equals the reference's."""
    g = _golden()["big"]
    w, h, D, seed = GW.BIG
    pairs = [T.synthetic_pair(w, h, D, seed + i) for i in range(12)]
    assert [T.sha(pairs[0][0]), T.sha(pairs[0][1])] == g["input_sha"]
    assert 12 * h * w * D > 2 ** 31
    eng = _engine(w, h, T.default_option(max_disparity=D), wave_pairs=12, lanes=1, max_disparity_range=WIDE)
    assert eng.wave_pairs == 12
    batch = eng.match_batch(np.stack([p[0] for p in pairs]), np.stack([p[1] for p in pairs]))
    assert T.sha(batch[0]) == g["final_sha"], "seed 1 differs from the reference"
    for i, (l, r) in enumerate(pairs):
        _same(f"pair {i}", batch[i], eng.match(l, r))
    eng.close()


@pytest.mark.gpu
def test_limits_on_gpu(cone):
    """512 runs and the resolved limit is reported; the default stays 256; a Cone engine with the wide limit computes the
    reference's Cone map; the Python class keeps its limit through Reset."""
    import adcensus_b200 as A
    w, h = 64, 40
    opt = T.default_option(max_disparity=WIDE)
    left, right = T.synthetic_pair(w, h, WIDE, 50)
    eng = _engine(w, h, opt, max_disparity_range=WIDE)
    _same("D = 512", eng.match(left, right), T.Oracle(w, h, opt).match(left, right))
    eng.close()
    eng = _engine(w, h, T.default_option(max_disparity=300), max_disparity_range=300)
    assert eng.max_disparity_range == 300
    eng.close()
    eng = _engine(w, h, T.default_option(max_disparity=16))
    assert eng.max_disparity_range == 256
    eng.close()
    cl, cr = cone
    ch, cw, _ = cl.shape
    eng = _engine(cw, ch, T.default_option(), max_disparity_range=WIDE)
    want = json.loads(str(np.load(T.GOLDEN_DIR / "golden_cone_full.npz")["hashes"]))["MEDIAN/DISP_L"]
    assert T.sha(eng.match(cl, cr)) == want
    eng.close()
    s = A.ADCensusStereo()
    o = A.ADCensusOption(max_disparity=400)
    assert s.Initialize(w, h, o) is False and "disparity range" in s.last_error
    assert s.Initialize(w, h, o, max_disparity_range=WIDE) is True
    assert s.Reset(w, h, o) is True
    assert s.Match(np.zeros((h, w, 3), np.uint8), np.zeros((h, w, 3), np.uint8)).shape == (h, w)
    s.Release()


@pytest.mark.gpu
def test_cpp_wide_overload_on_gpu(tmp_path):
    """tests/cpp/wide_main.cpp: the C++ class with Initialize(width, height, option, 512) at D = 400; its map against
    the oracle."""
    import adcensus_b200 as A
    exe = tmp_path / "wide"
    r = subprocess.run(["g++", "-std=c++17", str(T.REPO / "tests" / "cpp" / "wide_main.cpp"), f"-I{T.REPO / 'include'}",
                        f"-L{A.lib_path().parent}", "-ladcensus_b200", f"-Wl,-rpath,{A.lib_path().parent}", "-o", str(exe)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    w, h, D = 320, 40, 400
    left, right = T.synthetic_pair(w, h, D, 42)
    left.tofile(tmp_path / "left.bgr"); right.tofile(tmp_path / "right.bgr")
    run = subprocess.run([str(exe), str(tmp_path / "left.bgr"), str(tmp_path / "right.bgr"), str(w), str(h), "0", str(D),
                          str(tmp_path / "disp.f32")], capture_output=True, text=True, env=dict(os.environ, ADC_B200_QUIET="1"))
    assert run.returncode == 0 and "WIDE_OK" in run.stdout, (run.returncode, run.stdout[-500:], run.stderr[-500:])
    got = np.fromfile(tmp_path / "disp.f32", np.float32).reshape(h, w)
    _same("C++ D = 400", got, T.Oracle(w, h, T.default_option(max_disparity=D)).match(left, right))
